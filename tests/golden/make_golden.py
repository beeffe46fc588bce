#!/usr/bin/env python3
"""Regenerates the committed fixtures under tests/golden/.  Run in the build container (needs /root/reference for the
reference-derived fixtures and the oracle for the generated vectors):  python tests/golden/make_golden.py

  single_div_nondet.machine.json   machine section of /root/reference/autoprecompiles/tests/single_div_nondet.json.gz
  wasm_register_reuse.machine.json machine section of .../wasm_register_reuse.json.gz
  apc_reth_op_bug.machine.json.gz  machine section of .../apc_reth_op_bug.json.gz: a real PRE-optimisation APC (5869 columns,
                                   9168 constraints, 3117 bus interactions) -- the large-AIR case for the compiler, the
                                   interpreter and the chunked JIT
  apc_snapshots.json               the 62 optimized machines of /root/reference/openvm-riscv/tests/apc_snapshots/**
                                   re-serialised in the reference JSON expression schema (constraints + bus interactions)
  fixture_stats.json               sizes/degree histograms of the big reference fixtures (keccak/sha256/ecrecover ...)
  oracle_kat.json                  known-answer vectors produced BY THE ORACLE (Poseidon2, sponge, compress, challenger,
                                   small LDE / fold) -- regression pins for oracle and GPU alike
  segment_2p8_w12.json             a whole-segment proof produced by the oracle
  segment_logup_2p7.json           the same with bus interactions (LogUp phase, transcript v2): proof + digests of the opened values / queries
  stage0_subs.json.gz              instruction opcodes + per-instruction substitution tables (`block`, `subs` sections) of
                                   single_div_nondet, wasm_register_reuse and keccak_apc_pre_opt (677 instructions, 27 521 cells): the
                                   REAL stage-0 gather pattern (the machines of the big fixture are not committed: 28 627 constraints)
  chips_mixed.json                 three chips of different heights under one transcript (orc_prove_chips): proof, cumulative sums, digests
  v1_metrics.json                  the OpenVM-1 metrics document powdr_b200.metrics writes for one segment, and the summary the
                                   reference's own tooling (openvm-riscv/scripts/basic_metrics.py extract_metrics) reads from it
"""
import glob
import gzip
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import orc  # noqa: E402
from powdr_b200 import machine as M  # noqa: E402
from util import rand_field  # noqa: E402

REF = "/root/reference"


def dump(name, obj):
    with open(os.path.join(HERE, name), "w") as f:
        json.dump(obj, f, separators=(",", ":"))
    print("wrote", name, os.path.getsize(os.path.join(HERE, name)), "bytes")


def main():
    if os.path.isdir(REF):
        for name in ("single_div_nondet", "wasm_register_reuse"):
            doc = json.load(gzip.open(os.path.join(REF, "autoprecompiles/tests/%s.json.gz" % name), "rt"))
            dump(name + ".machine.json", {"machine": doc["machine"], "bus_map": doc.get("bus_map")})
        doc = json.load(gzip.open(os.path.join(REF, "autoprecompiles/tests/apc_reth_op_bug.json.gz"), "rt"))
        with gzip.GzipFile(os.path.join(HERE, "apc_reth_op_bug.machine.json.gz"), "wb", mtime=0) as f:      # 5869 columns, 9168 constraints
            f.write(json.dumps({"machine": doc["machine"], "bus_map": doc.get("bus_map")}, separators=(",", ":")).encode())
        snaps = {}
        for p in sorted(glob.glob(os.path.join(REF, "openvm-riscv/tests/apc_snapshots/*/*.txt"))):
            mach = M.SymbolicMachine.from_snapshot_text(open(p).read())
            key = os.path.relpath(p, os.path.join(REF, "openvm-riscv/tests/apc_snapshots"))
            snaps[key] = {"columns": mach.snapshot_columns, "constraints": mach.constraints, "bus_interactions": mach.bus_interactions}
        dump("apc_snapshots.json", snaps)
        stats = {}
        for name in ("keccak_apc_pre_opt", "ecrecover_apc_pre_opt", "sha256_apc_pre_opt", "single_div_nondet", "apc_reth_op_bug"):
            doc = json.load(gzip.open(os.path.join(REF, "autoprecompiles/tests/%s.json.gz" % name), "rt"))
            mach = M.SymbolicMachine(doc["machine"]["constraints"], doc["machine"]["bus_interactions"], doc["machine"]["derived_columns"])
            hist = [0, 0, 0, 0]
            for c in mach.constraints:
                hist[M.degree(c)] += 1
            stats[name] = {"columns": mach.width, "constraints": len(mach.constraints), "bus_interactions": len(mach.bus_interactions),
                           "degree_hist": hist}
        dump("fixture_stats.json", stats)
        st0 = {}
        for name in ("single_div_nondet", "wasm_register_reuse", "keccak_apc_pre_opt"):
            doc = json.load(gzip.open(os.path.join(REF, "autoprecompiles/tests/%s.json.gz" % name), "rt"))
            mach = M.SymbolicMachine(doc["machine"]["constraints"], doc["machine"]["bus_interactions"], doc["machine"]["derived_columns"])
            assert mach.column_ids == list(range(mach.width)), name           # pre-opt machines: contiguous poly ids, all used
            ops = [ins[0] for b in doc["block"]["blocks"] for ins in b["instructions"]]
            subs = [[[s_["original_poly_index"], s_["apc_poly_id"]] for s_ in ss] for ss in doc["subs"]]
            assert len(ops) == len(subs)
            st0[name] = {"n_columns": mach.width, "opcodes": ops, "subs": subs}
        with gzip.GzipFile(os.path.join(HERE, "stage0_subs.json.gz"), "wb", mtime=0) as f:
            f.write(json.dumps(st0, separators=(",", ":")).encode())
        print("wrote stage0_subs.json.gz", os.path.getsize(os.path.join(HERE, "stage0_subs.json.gz")), "bytes")
        v1_metrics()
    rng = np.random.default_rng(2024)
    kat = {}
    kat["perm_zero"] = orc.poseidon2_permute(np.zeros(16, dtype=np.uint32)).tolist()
    st = np.arange(16, dtype=np.uint32)
    kat["perm_iota"] = orc.poseidon2_permute(st).tolist()
    row = rand_field(rng, 21)
    kat["row21"] = row.tolist()
    kat["hash_row21"] = orc.hash_row(row).tolist()
    kat["compress"] = orc.compress(np.arange(8, dtype=np.uint32), np.arange(8, 16, dtype=np.uint32)).tolist()
    ch = orc.Challenger()
    ch.observe(np.arange(1, 12, dtype=np.uint32))
    kat["challenger_after_11"] = [ch.sample() for _ in range(10)]
    tr = rand_field(rng, (2, 8))
    kat["lde_in"] = tr.tolist()
    kat["lde_out"] = orc.lde_batch(tr, 1, 31).tolist()
    f = rand_field(rng, (8, 4))
    beta = rand_field(rng, 4)
    kat["fold_in"], kat["fold_beta"] = f.tolist(), beta.tolist()
    kat["fold_out"] = orc.fri_fold(f, 31, beta).tolist()
    dump("oracle_kat.json", kat)

    g = {"width": 12, "n_constraints": 5, "seed": 8, "trace_seed": 4242, "log_n": 8}
    mach = M.synthetic_machine(g["width"], g["n_constraints"], seed=g["seed"])
    bc, spans = M.compile_constraints(mach)
    trace = rand_field(np.random.default_rng(g["trace_seed"]), (mach.width, 1 << g["log_n"]))
    g["proof"], _ = orc.prove_segment(trace, bc, spans)
    dump("segment_2p8_w12.json", g)

    import hashlib
    sha = lambda a: hashlib.sha256(np.ascontiguousarray(a, dtype=np.uint32).tobytes()).hexdigest()
    g = {"width": 14, "n_constraints": 4, "n_interactions": 9, "quadratic_every": 4, "seed": 21, "bus_seed": 22, "trace_seed": 777, "log_n": 7,
         "n_queries": 8, "pow_bits": 4}
    base = M.synthetic_machine(g["width"], g["n_constraints"], seed=g["seed"])
    mach = M.SymbolicMachine(base.constraints, M.synthetic_bus(base, g["n_interactions"], g["bus_seed"], g["quadratic_every"]))
    bc, spans = M.compile_constraints(mach)
    trace = rand_field(np.random.default_rng(g["trace_seed"]), (mach.width, 1 << g["log_n"]))
    proof, ys, q, _ = orc.prove(trace, bc, spans, M.compile_bus(mach, 1), n_queries=g["n_queries"], pow_bits=g["pow_bits"])
    g.update(proof=proof, ys_sha256=sha(ys), queries_sha256=sha(q))
    dump("segment_logup_2p7.json", g)

    g = {"spec": [[6, 12, 3, 7], [4, 9, 2, 0], [3, 10, 0, 3]], "seed": 5, "n_queries": 6, "pow_bits": 5}
    chips = chips_for(g["spec"], g["seed"])
    proof, cs, ys, q = orc.prove_chips(chips, n_queries=g["n_queries"], pow_bits=g["pow_bits"])
    g.update(proof=proof, cumsums=cs.tolist(), ys_sha256=sha(ys), queries_sha256=sha(q))
    dump("chips_mixed.json", g)


def v1_metrics():
    """one segment's stage times through powdr_b200.metrics, then through the reference's basic_metrics.extract_metrics (its
    matplotlib import serves the plots only and is stubbed where matplotlib is not installed)"""
    import tempfile
    import types
    from powdr_b200 import metrics
    inputs = {"stage_ms": {"h2d": 0.1, "lde": 34.0, "merkle": 130.0, "logup_gen": 46.0, "logup_commit": 270.0, "quotient": 60.0, "qlde": 0.3,
                           "qmerkle": 1.3, "open": 25.0, "fri": 3.9, "pow": 0.3, "total": 571.0},
              "rows": 1 << 20, "main_cols": 2022, "perm_cols": 3348, "n_constraints": 187, "n_interactions": 1734, "trace_gen_ms": 12.0, "query_ms": 0.5}
    doc = metrics.segment_metrics(inputs["stage_ms"], inputs["rows"], inputs["main_cols"], inputs["perm_cols"], inputs["n_constraints"],
                                  inputs["n_interactions"], trace_gen_ms=inputs["trace_gen_ms"], query_ms=inputs["query_ms"])
    try:
        import matplotlib  # noqa: F401
    except ImportError:
        mpl = types.ModuleType("matplotlib")
        mpl.pyplot, mpl.ticker = types.ModuleType("matplotlib.pyplot"), types.ModuleType("matplotlib.ticker")
        mpl.ticker.AutoMinorLocator = None
        sys.modules.update({"matplotlib": mpl, "matplotlib.pyplot": mpl.pyplot, "matplotlib.ticker": mpl.ticker})
    sys.path.insert(0, os.path.join(REF, "openvm-riscv/scripts"))
    import basic_metrics
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "metrics.json")
        metrics.write(path, doc)
        out = basic_metrics.extract_metrics(path)
    summary = {k: (float(v) if isinstance(v, float) else int(v)) for k, v in out.items() if k != "filename"}
    dump("v1_metrics.json", {"inputs": inputs, "metrics": doc, "basic_metrics": summary})


def chips_for(spec, seed):
    """[(log_n, width, n_constraints, n_interactions)] -> [(trace, bytecode, spans, bus)]; shared with tests/test_oracle_chips.py"""
    rng = np.random.default_rng(seed)
    out = []
    for i, (log_n, width, ncons, nints) in enumerate(spec):
        base = M.synthetic_machine(width, ncons, seed=100 + i) if ncons else None
        bus_json = M.synthetic_bus(width, nints, seed=200 + i, quadratic_every=5) if nints else []
        mach = M.SymbolicMachine(base.constraints if base else [], bus_json)
        bc, spans = M.compile_constraints(mach)
        out.append((rand_field(rng, (mach.width, 1 << log_n)), bc, spans, M.compile_bus(mach, 1) if nints else None))
    return out


if __name__ == "__main__":
    main()
