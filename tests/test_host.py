"""CPU tests of the host side: machine loader / bytecode compiler (mirror of emit_expr), the C-ABI library exporting every
symbol the header declares, and loud failure without a GPU."""
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def test_library_exports_every_declared_symbol():
    import powdr_b200
    from powdr_b200 import build, capi
    build.build()
    lib = powdr_b200.load_library()
    header = open(os.path.join(ROOT, "include", "powdr_b200.h")).read()
    declared = set(re.findall(r"^(?:int|uint64_t)\s+(\w+)\(", header, flags=re.M))
    assert len(declared) >= 28
    for name in declared:
        assert hasattr(lib, name), name
    assert declared == set(capi.EXPORTS)


def test_no_cpu_fallback_without_gpu():
    import powdr_b200
    from powdr_b200.capi import PbError
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("GPU present")
    except ImportError:
        pass
    with pytest.raises(PbError) as e:
        powdr_b200.Context(0)
    assert e.value.code == -5


def test_column_order_is_ascending_poly_id():
    from powdr_b200 import machine as M
    mach = M.SymbolicMachine([["b@7", "*", "a@3"], ["c@11", "-", "a@3"]])
    assert mach.column_ids == [3, 7, 11] and mach.width == 3
    bc, spans = M.compile_constraints(mach)
    assert bc == [0, 1, 0, 0, 4, 0, 2, 0, 0, 3] and spans == [(0, 5), (5, 5)]


def test_derived_and_bus_compilers_follow_reference_layout():
    from powdr_b200 import machine as M
    mach = M.SymbolicMachine(
        [["x@0", "*", "y@1"]],
        [{"id": 3, "mult": "x@0", "args": [["y@1", "+", 1], 17]}],
        [["z@2", {"QuotientOrZero": ["x@0", "y@1"]}], ["k@3", {"Constant": 9}]])
    H = 16
    specs, bc = M.compile_derived(mach, H)
    # denominator, INV_OR_ZERO, numerator, MUL (cuda/mod.rs:124-130); PUSH_APC operand = col*H (cuda/mod.rs:61)
    assert bc[:6] == [0, 1 * H, 6, 0, 0 * H, 4] and specs[0] == (2, 0, 6)
    assert bc[6:] == [1, 9] and specs[1] == (3, 6, 2)
    ints, spans, bbc = M.compile_bus(mach, H)
    assert ints == [(3, 2, 0)] and len(spans) == 3        # [mult, arg0, arg1] (cuda_abi.rs:150-160)
    assert bbc[spans[0][0]:spans[0][0] + spans[0][1]] == [0, 0]
    assert bbc[spans[2][0]:spans[2][0] + spans[2][1]] == [1, 17]


def test_periphery_bus_ids_come_from_the_fixture_bus_map():
    """the bus ids / tuple-checker sizes the histogram kernel is called with (cuda/mod.rs:359-372) read from the `bus_map` of the reference
    fixtures; they are also the defaults of `Context.bus_compile` / `_apc_apply_bus` callers here"""
    import json
    from powdr_b200 import machine as M
    a = json.load(open(os.path.join(GOLDEN, "single_div_nondet.machine.json")))
    assert M.periphery_from_bus_map(a["bus_map"]) == {"var_bus": 3, "bitwise_bus": 6, "tuple2_bus": 7, "tuple2_sizes": (256, 2048)}
    b = json.load(open(os.path.join(GOLDEN, "wasm_register_reuse.machine.json")))
    assert M.periphery_from_bus_map(b["bus_map"])["tuple2_sizes"] == (256, 4096)
    assert M.periphery_from_bus_map(None)["var_bus"] is None


def test_stack_depth_of_fixtures_fits_reference_capacity():
    from powdr_b200 import machine as M
    mach = M.SymbolicMachine.from_json_file(os.path.join(GOLDEN, "single_div_nondet.machine.json"))
    bc, spans = M.compile_constraints(mach)
    worst = 0
    for off, ln in spans:
        d, ip = 0, off
        while ip < off + ln:
            op = bc[ip]
            ip += 1
            if op in (0, 1):
                ip += 1
                d += 1
            elif op in (2, 3, 4):
                d -= 1
            worst = max(worst, d)
    assert worst <= 16 and worst == 7      # SURVEY.md App. A: max eval-stack depth 7 for this fixture


def test_synthetic_machine_shape():
    from powdr_b200 import machine as M
    mach = M.synthetic_machine(2022, 187, seed=1)
    assert mach.width == 2022 and len(mach.constraints) == 187
    assert max(M.degree(c) for c in mach.constraints) == 3


def test_jit_codegen_compiles_for_sm100a_without_a_device():
    """pb_air_jit_compile_only: pack the reference fixture's constraints, generate CUDA C, NVRTC-compile for sm_100a"""
    import ctypes as C
    import powdr_b200
    from powdr_b200 import machine as M
    from powdr_b200.capi import Span
    lib = powdr_b200.load_library()
    mach = M.SymbolicMachine.from_json_file(os.path.join(GOLDEN, "single_div_nondet.machine.json"))
    bc, spans = M.compile_constraints(mach)
    b = np.array(bc, dtype=np.uint32)
    sp = (Span * len(spans))()
    for i, (o, l) in enumerate(spans):
        sp[i].off, sp[i].len = o, l
    sz = C.c_size_t()
    rc = lib.pb_air_jit_compile_only(b.ctypes.data_as(C.c_void_p), C.c_size_t(b.size), sp, C.c_size_t(len(spans)), C.c_uint32(mach.width), C.byref(sz))
    assert rc == 0 and sz.value > 1000
    # malformed program is rejected before any code generation
    bad = np.array([0, 99], dtype=np.uint32)
    sp1 = (Span * 1)()
    sp1[0].off, sp1[0].len = 0, 2
    assert lib.pb_air_jit_compile_only(bad.ctypes.data_as(C.c_void_p), C.c_size_t(2), sp1, C.c_size_t(1), C.c_uint32(3), C.byref(sz)) == -4


def test_shard_columns_partition():
    """pb_shard_columns: contiguous blocks of ceil(W/G) columns, trailing ranks may be short or empty; no GPU needed"""
    from powdr_b200.sharded import shard_columns
    for width, world in [(2022, 8), (2022, 2), (12, 8), (5, 8), (256, 4), (1, 2)]:
        blocks = [shard_columns(width, world, r) for r in range(world)]
        per = -(-width // world)
        assert all(c <= per for _, c in blocks)
        cols = [c for f, n in blocks for c in range(f, f + n)]
        assert cols == list(range(width))


def test_comm_struct_wraps_python_callables():
    from powdr_b200.sharded import Comm, PbComm
    calls = []

    class Rec(Comm):
        def all_gather(self, send, recv, nbytes):
            calls.append(("ag", send, recv, nbytes))

        def all_to_all(self, send, recv, nbytes):
            raise RuntimeError("boom")

    c = Rec(1, 4)
    assert isinstance(c.c, PbComm) and c.c.rank == 1 and c.c.world == 4
    assert c.c.all_gather(None, 16, 32, 8) == 0 and calls == [("ag", 16, 32, 8)]
    assert c.c.all_to_all(None, 0, 0, 0) == 1 and isinstance(c.error, RuntimeError)     # exceptions never cross into C


def test_header_is_plain_c_and_cxx(tmp_path):
    """include/powdr_b200.h is the drop-in boundary: it must compile as C99 and as C++ with nothing but the standard headers"""
    import subprocess
    hdr = os.path.join(ROOT, "include")
    c = tmp_path / "t.c"
    c.write_text('#include "powdr_b200.h"\nint main(void) { pb_segment_proof_t p; pb_comm_t c; (void)p; (void)c; return PB_ERR_COMM == -6 ? 0 : 1; }\n')
    subprocess.check_call(["/usr/bin/gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-fsyntax-only", "-I", hdr, str(c)])
    cc = tmp_path / "t.cc"
    cc.write_text(c.read_text())
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-Wall", "-Werror", "-fsyntax-only", "-I", hdr, str(cc)])


def test_product_never_imports_the_oracle():
    """oracle/ is test infrastructure: nothing under powdr_b200/ (python or CUDA) may reference it"""
    pkg = os.path.join(ROOT, "powdr_b200")
    for dirpath, _, files in os.walk(pkg):
        if "_lib" in dirpath or "__pycache__" in dirpath:
            continue
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".inl", ".h")):
                txt = open(os.path.join(dirpath, f), errors="replace").read()
                assert "import oracle" not in txt and "from oracle" not in txt and "oracle/" not in txt.replace("the oracle/", ""), f


def test_logup_codegen_compiles_for_sm100a_without_a_device():
    """host-only check of the LogUp generator (pb_air_logup_compile_only): chunking by the degree rule, generated CUDA C for the
    permutation-trace and the fold kernels accepted by NVRTC for sm_100a; malformed interaction tables are rejected"""
    import ctypes as C
    import numpy as np
    import powdr_b200
    from powdr_b200 import machine as M, capi
    lib = powdr_b200.load_library()
    mach = M.SymbolicMachine([], M.synthetic_bus(24, 21, 3, quadratic_every=5))
    ints, isp, ibc = M.compile_bus(mach, 1)
    ibc = np.array(ibc, dtype=np.uint32)
    spn = (capi.Span * len(isp))()
    for i, (o, l) in enumerate(isp):
        spn[i].off, spn[i].len = o, l
    di = (capi.DevInteraction * len(ints))()
    for i, (b, n, o) in enumerate(ints):
        di[i].bus_id, di[i].num_args, di[i].args_index_off = b, n, o
    cb, wp = C.c_size_t(), C.c_size_t()
    args = (ibc.ctypes.data_as(C.c_void_p), C.c_size_t(ibc.size), spn, C.c_size_t(len(isp)), di, C.c_size_t(len(ints)), C.c_uint32(mach.width))
    assert lib.pb_air_logup_compile_only(*args, C.byref(cb), C.byref(wp)) == 0
    # 21 interactions, every 5th with a degree-2 argument (own chunk): 4 singles + ceil-pairs of the runs of 4 -> 4 + 4*2 + 1 = 13 chunks
    assert wp.value == 4 * (13 + 1) and cb.value > 10000
    # the generated stage-0 periphery kernel compiles from the same table (ctx = out = NULL: host-only check)
    assert lib.pb_bus_compile(None, *args, C.c_uint32(3), C.c_uint32(7), C.c_uint32(6), None) == 0
    di[3].args_index_off = len(isp)              # spans out of range
    assert lib.pb_air_logup_compile_only(*args, C.byref(cb), C.byref(wp)) == -4
    assert lib.pb_bus_compile(None, *args, C.c_uint32(3), C.c_uint32(7), C.c_uint32(6), None) == -4


def test_chunked_jit_compiles_a_9168_constraint_machine_in_parallel():
    """the real pre-optimisation fixture is 141 k bytecode words: as one NVRTC module that took 11 minutes, as 2 k-word chunks on
    all host threads it must stay a key-generation-time cost (seconds to tens of seconds)"""
    import ctypes as C
    import time
    import powdr_b200
    from powdr_b200 import machine as M
    from powdr_b200.capi import Span
    mach = M.SymbolicMachine.from_json_file(os.path.join(GOLDEN, "apc_reth_op_bug.machine.json.gz"))
    bc, spans = M.compile_constraints(mach)
    bc = np.ascontiguousarray(bc, dtype=np.uint32)
    sp = (Span * len(spans))()
    for i, (o, l) in enumerate(spans):
        sp[i].off, sp[i].len = o, l
    lib = powdr_b200.load_library()
    n = C.c_size_t()
    t0 = time.time()
    rc = lib.pb_air_jit_compile_only(bc.ctypes.data_as(C.c_void_p), C.c_size_t(bc.size), sp, C.c_size_t(len(spans)), C.c_uint32(mach.width), C.byref(n))
    assert rc == 0 and n.value > 1 << 20
    assert time.time() - t0 < 300


def _build_abi_demo(tmp_path):
    import subprocess
    exe = str(tmp_path / "abi_demo")
    lib_dir = os.path.join(ROOT, "powdr_b200", "_lib")
    subprocess.check_call(["/usr/bin/gcc", "-std=c99", "-O2", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "examples", "abi_demo.c"), "-L", lib_dir, "-lpowdr_b200", "-Wl,-rpath," + lib_dir, "-o", exe])
    return exe


def test_plain_c_client_links_and_fails_loudly_without_a_gpu(tmp_path):
    """examples/abi_demo.c uses nothing but the header and the .so; without a device pb_ctx_create must return PB_ERR_NO_DEVICE"""
    import subprocess
    import powdr_b200
    powdr_b200.load_library()
    r = subprocess.run([_build_abi_demo(tmp_path), "6"], capture_output=True, text=True, timeout=120)
    if r.returncode != 0:
        assert "pb_ctx_create" in r.stderr and "-> -5" in r.stderr, r.stderr
    else:                                   # a GPU is present where this CPU suite runs: the demo must then succeed
        assert "trace_root" in r.stdout


def test_bench_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (the CPU restatement timed on the host cores) needs no GPU and must print exactly one JSON line
    with the contract's keys"""
    import json
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", "--log-n", "12",
                        "--width", "24", "--constraints", "5", "--interactions", "9", "--queries", "10", "--pow-bits", "6"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["higher_is_better"] is False and d["value"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and "full configuration" in cb["sample"] and cb["stages_s"]["logup_gen"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]


def test_bench_reference_arm_under_torchrun_prints_once_from_rank_0():
    """the driver launches the reference arm like the native one at N > 1 (torchrun, one process per GPU): rank 0 alone times and prints,
    the other ranks exit 0 without work, no process group is needed"""
    import json
    import socket
    import subprocess
    import sys
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", str(port), os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0",
                        "--log-n", "10", "--width", "24", "--constraints", "5", "--interactions", "9", "--queries", "10", "--pow-bits", "6"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["value"] > 0 and d["cpu_baseline"]["kind"] == "port"


def test_entry_points_reject_null_arguments_before_touching_the_device():
    """error behaviour of the boundary (cuda_abi.rs convention: an int comes back, nothing aborts): every compute entry point
    returns PB_ERR_INVALID_ARG for null handles / pointers -- checked here without a GPU"""
    import ctypes as C
    import powdr_b200
    lib = powdr_b200.load_library()
    z, n0 = C.c_void_p(0), C.c_size_t(0)
    four = (C.c_uint32 * 4)(1, 2, 3, 4)
    INVALID = -1
    assert lib.pb_lde_batch(z, z, C.c_size_t(4), C.c_size_t(1), C.c_uint32(1), C.c_uint32(31), z) == INVALID
    assert lib.pb_quotient(z, z, z, C.c_size_t(4), C.c_uint32(1), C.c_uint32(31), four, z) == INVALID
    assert lib.pb_constraint_fold(z, z, z, C.c_size_t(4), four, z) == INVALID
    assert lib.pb_merkle_commit(z, z, z, n0, C.c_size_t(3), z, z) == INVALID
    assert lib.pb_merkle_commit_rows8(z, z, C.c_size_t(3), z, z) == INVALID
    assert lib.pb_fri_fold(z, z, C.c_size_t(4), C.c_uint32(31), four, z) == INVALID
    assert lib.pb_eval_at_point(z, z, C.c_size_t(4), C.c_size_t(1), C.c_uint32(1), four, z) == INVALID
    assert lib.pb_deep_quotient(z, z, z, n0, C.c_size_t(4), C.c_uint32(31), four, four, z, z) == INVALID
    assert lib.pb_prove_segment(z, z, z, C.c_size_t(4), C.c_size_t(1), C.c_uint32(0), z) == INVALID
    assert lib.pb_prove_segment_sharded(z, z, z, C.c_size_t(4), C.c_size_t(1), C.c_uint32(0), z, z) == INVALID
    assert lib.pb_lde_shard(z, z, C.c_size_t(6), C.c_size_t(1), C.c_uint32(31), C.c_int(2), C.c_int(0), z) == INVALID
    assert lib.pb_poseidon2_permute(z, z, n0, C.c_int(1)) == INVALID
    first, count = C.c_size_t(), C.c_size_t()
    assert lib.pb_shard_columns(C.c_size_t(10), C.c_int(4), C.c_int(4), C.byref(first), C.byref(count)) == INVALID      # rank out of range
    assert lib.pb_query_words(C.c_size_t(10), C.c_size_t(3), n0, z) == INVALID
    assert lib.pb_air_set_interactions(z, z, z, n0, z, n0, z, n0) == INVALID
    assert lib.pb_allgather_caps(z, z, z, z) == INVALID
    assert lib.pb_ctx_set_fri_params(z, C.c_uint32(8), C.c_uint32(4)) == INVALID
    assert lib.pb_prove_chips(z, z, C.c_size_t(1), z, z) == INVALID
    assert lib.pb_chips_sizes(z, C.c_size_t(1), z, z) == INVALID
    assert lib.pb_query_chips(z, z, n0, z, n0) == INVALID
    assert lib.pb_query_segment_sharded(z, z, z, n0) == INVALID


def test_v1_metrics_json_is_consumed_by_the_reference_tooling(tmp_path):
    """SURVEY §8 f4: the per-stage times go out under the OpenVM-1 metric names.  tests/golden/v1_metrics.json holds the document
    written for these stage times and the summary the reference's own basic_metrics.extract_metrics read from it
    (tests/golden/make_golden.py); the writer must still produce that document, byte for byte after parsing"""
    import json
    from powdr_b200 import metrics
    gold = json.load(open(os.path.join(GOLDEN, "v1_metrics.json")))
    inp = gold["inputs"]
    m = metrics.segment_metrics(inp["stage_ms"], inp["rows"], inp["main_cols"], inp["perm_cols"], inp["n_constraints"], inp["n_interactions"],
                                trace_gen_ms=inp["trace_gen_ms"], query_ms=inp["query_ms"])
    path = tmp_path / "metrics.json"
    metrics.write(str(path), m)
    doc = json.load(open(path))
    names = {g["metric"] for g in doc["gauge"]}
    for k in ("main_trace_commit_time_ms", "perm_trace_commit_time_ms", "quotient_poly_compute_time_ms", "quotient_poly_commit_time_ms",
              "pcs_opening_time_ms", "stark_prove_excluding_trace_time_ms", "total_proof_time_ms", "trace_gen_time_ms"):
        assert k in names
    assert doc == gold["metrics"]
    out = gold["basic_metrics"]
    assert out["num_segments"] == 1 and out["powdr_ratio"] == 1.0 and out["powdr_rows"] == 1 << 20
    assert abs(out["app_proof_time_excluding_trace_ms"] - 571.5) < 1e-6 and out["app_proof_cols"] == 2022 + 3348


def test_host_transcript_permutation_kat_and_simd_equals_scalar():
    """the host side of the transcript (AVX-512 when the CPU has it) against the Plonky3 known answer, the scalar version, and the
    oracle's permutation on random states"""
    import ctypes as C
    import powdr_b200
    from oracle import orc
    orc.build()
    lib = powdr_b200.load_library()
    used = C.c_int(-1)
    st = (C.c_uint32 * 16)(*range(16))
    assert lib.pb_host_poseidon2_permute(st, 1, 0, C.byref(used)) == 0
    kat = [1906786279, 1737026427, 1959749225, 700325316]
    assert list(st)[:4] == kat and st[15] == 304856115
    st2 = (C.c_uint32 * 16)(*range(16))
    assert lib.pb_host_poseidon2_permute(st2, 1, 1, None) == 0 and list(st2) == list(st)
    rng = np.random.default_rng(5)
    for reps in (1, 2, 7):
        s = rng.integers(0, 2013265921, 16, dtype=np.uint32)
        a, b = (C.c_uint32 * 16)(*s.tolist()), (C.c_uint32 * 16)(*s.tolist())
        assert lib.pb_host_poseidon2_permute(a, reps, 0, None) == 0 and lib.pb_host_poseidon2_permute(b, reps, 1, None) == 0
        exp = s.copy()
        for _ in range(reps):
            exp = np.asarray(orc.poseidon2_permute(exp), dtype=np.uint32)
        assert list(a) == list(b) == exp.tolist()
    assert lib.pb_host_poseidon2_permute(None, 1, 0, None) == -1
    assert used.value in (0, 1)


def test_host_transcript_generic_diagonal_branch(tmp_path):
    """tests/host_transcript_check.cpp: AVX-512 vs scalar host permutation with a non-default internal diagonal, 50 k chained permutations"""
    import subprocess
    exe = str(tmp_path / "htc")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-o", exe, os.path.join(ROOT, "tests", "host_transcript_check.cpp"),
                           os.path.join(ROOT, "powdr_b200", "csrc", "transcript_host.cpp")])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "bad=0" in r.stdout, r.stdout + r.stderr


def test_bench_dump_outputs_is_exact_and_capped(tmp_path, monkeypatch):
    """bench.py --dump-outputs: field elements and 32-bit words survive the float64 files exactly; above the size cap a fixed,
    seeded sample of the query rows is written together with its row indices"""
    import sys
    sys.path.insert(0, ROOT)
    import bench
    proof = {"trace_root": list(range(8)), "fri_roots": [[7] * 8] * 3, "final_poly": [], "pow_witness": 2**32 - 1}
    q = np.random.default_rng(1).integers(0, 2**32, (100, 500), dtype=np.uint32)
    ys = np.arange(40, dtype=np.uint32).reshape(10, 4)
    bench.dump_outputs(str(tmp_path / "all"), proof, {"queries": q, "opened_values": ys})
    assert (np.load(tmp_path / "all" / "queries.npy") == q).all() and (np.load(tmp_path / "all" / "opened_values.npy") == ys).all()
    assert np.load(tmp_path / "all" / "pow_witness.npy") == 2**32 - 1 and np.load(tmp_path / "all" / "fri_roots.npy").shape == (3, 8)
    assert not (tmp_path / "all" / "query_rows.npy").exists()
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 1 << 17)
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), proof, {"queries": q, "opened_values": ys})
        assert sum(f.stat().st_size - 128 for f in (tmp_path / d).iterdir()) <= 1 << 17        # .npy header: 128 bytes
    rows = np.load(tmp_path / "s1" / "query_rows.npy").astype(np.int64)
    assert 0 < len(rows) < 100 and (np.load(tmp_path / "s1" / "queries.npy") == q[rows]).all()
    assert (rows == np.load(tmp_path / "s2" / "query_rows.npy")).all()
