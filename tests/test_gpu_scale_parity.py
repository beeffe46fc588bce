"""Bit-exact GPU parity at the sizes where the specialised kernels run (2^16 - 2^24 rows), against the AVX-512 CPU arm of the oracle
(oracle/fast.c, pinned to the scalar oracle at these sizes by tests/test_oracle_fast.py).

The verifier and the sampled checks of test_gpu_fullsize.py cannot see a kernel that commits self-consistently to the wrong thing: a
wrong coset or twiddle in one size-specific NTT pass, a wrong leaf hash at a row no query opens, a wrong LogUp column that the fold
kernel mirrors.  Each of those still gives a proof that verifies; here every LDE element, every Merkle node and every word of the
proof and its query openings is compared.  A failure names the first point of divergence and, for an LDE element or a Merkle node,
re-evaluates it with the scalar oracle to say which side is wrong.

Without AVX-512 on the host, the scalar oracle stands in where it takes well under a minute; the larger proofs are skipped."""
import ctypes as C

import numpy as np
import pytest

from util import P, rand_field, root_of_unity, structured_columns, lde_mismatch, merkle_mismatch, proof_mismatch

pytestmark = pytest.mark.gpu


def _fast(orc, scalar_ok):
    """True: compare against the AVX-512 arm; False: against the scalar oracle; skip when neither is practical"""
    if orc.fast_available():
        return True
    if not scalar_ok:
        pytest.skip("host CPU has no AVX-512 and the scalar oracle needs minutes at this size")
    return False


def _w2n_inv(log_n):
    """shift of the second quotient chunk's LDE (oracle/prove.c): 1 / w_{2N}"""
    return pow(root_of_unity(log_n + 1), P - 2, P)


def _batch(log_n):
    """LDE column batch of pb_lde_batch (lde_column_batch in csrc/capi.cu): 148 SMs x 16 tiles of 2^15 elements"""
    return 148 * 16 // max(1, (1 << log_n) >> 15)


# ---------------------------------------------------------------- a. LDE: every fast geometry, both cosets, every dispatch knob
KNOBS = {"": {}, "generic": {"PB_LDE_GENERIC": "1"}, "no_tma": {"PB_LDE_NO_TMA": "1"}, "batch3": {"PB_LDE_BATCH": "3"},
         "streams4": {"PB_LDE_STREAMS": "4"}}


def _lde_cases():
    out = []
    for log_n in range(18, 25):
        for knob in ("", "generic", "batch3", "streams4") + (("no_tma",) if log_n in (19, 20) else ()):
            out.append((log_n, 1, 31, knob))
        if log_n in (20, 22):
            out += [(log_n, 1, 1, ""), (log_n, 1, "w2n_inv", "")]
    for log_n in (18, 20):
        for log_blowup in (2, 3):
            out += [(log_n, log_blowup, 31, ""), (log_n, log_blowup, 31, "no_tma")]
    return out


_lde_ref = {}          # one entry: the cases of one (log_n, blowup, shift) are adjacent, the next one replaces it


def _lde_reference(orc, log_n, log_blowup, shift):
    key = (log_n, log_blowup, shift)
    if key not in _lde_ref:
        _lde_ref.clear()
        # width = batch + 1 at blowup 2 (two batches at every size: 297 columns at 2^18, 75 at 2^20, 5 at 2^24); narrower at the
        # larger blowups, which write 4 / 8 cosets per column
        width = _batch(log_n) + 1 if log_blowup == 1 else max(7, _batch(log_n) // 8 + 1)
        trace = structured_columns(np.random.default_rng(0x5CA1E + log_n), 1 << log_n, width)
        lde = (orc.fast_lde_batch if _fast(orc, True) else orc.lde_batch)(trace, log_blowup, shift)
        _lde_ref[key] = (trace, lde)
    return _lde_ref[key]


@pytest.mark.parametrize("log_n,log_blowup,shift,knob", _lde_cases())
def test_lde_equals_cpu_arm(ctx, orc, monkeypatch, log_n, log_blowup, shift, knob):
    shift = _w2n_inv(log_n) if shift == "w2n_inv" else shift
    trace, exp = _lde_reference(orc, log_n, log_blowup, shift)
    for k, v in KNOBS[knob].items():
        monkeypatch.setenv(k, v)
    width, n = trace.shape
    d_in = ctx.to_device(trace)
    d_out = ctx.alloc(exp.nbytes)
    ctx.lde_batch(d_in.ptr, log_n, width, d_out.ptr, log_blowup, shift)
    d_in.free()
    got = ctx.to_host(d_out, exp.shape)
    d_out.free()
    bad = lde_mismatch(got, exp, trace, log_blowup, shift)
    assert bad is None, "%s (knob %r): %s" % ((log_n, log_blowup, shift), knob, lde_mismatch(got, exp, trace, log_blowup, shift, orc))


# ---------------------------------------------------------------- b. Merkle: every layer (compress_block_kernel folds 10 levels per CTA from 2^20 nodes)
def _gpu_merkle(ctx, mats, log_h):
    h = 1 << log_h
    d_mats = [ctx.to_device(m) for m in mats]
    d_layers = ctx.alloc(32 * (2 * h))
    root = ctx.merkle_commit([d.ptr for d in d_mats], [m.shape[0] for m in mats], log_h, d_layers.ptr)
    flat = ctx.to_host(d_layers, (2 * h - 1, 8))        # digests are kept in Montgomery form on the device
    for d in d_mats:
        d.free()
    d_layers.free()
    layers, off, k = [], 0, h
    while k >= 1:
        layers.append(flat[off:off + k])
        off += k
        k >>= 1
    return root, layers


@pytest.mark.parametrize("log_h", [17, 19, 21])
@pytest.mark.parametrize("widths", [[8], [40], [9], [4, 4]], ids=["w8", "w40", "w9", "w4+4"])
def test_merkle_every_layer_equals_cpu_arm(ctx, orc, widths, log_h):
    rng = np.random.default_rng(log_h * 100 + sum(widths))
    mats = [rand_field(rng, (w, 1 << log_h)) for w in widths]
    exp = (orc.fast_merkle_commit if _fast(orc, True) else orc.merkle_commit)(mats)
    root, got = _gpu_merkle(ctx, mats, log_h)
    assert merkle_mismatch(got, exp, mats) is None, merkle_mismatch(got, exp, mats, orc)
    assert root == exp[-1][0].tolist()


def test_merkle_rows8_equals_cpu_arm(ctx, orc):
    log_h = 18
    rows = rand_field(np.random.default_rng(18), (1 << log_h, 8))
    mats = [np.ascontiguousarray(rows.T)]
    exp = (orc.fast_merkle_commit if _fast(orc, True) else orc.merkle_commit)(mats)
    d = ctx.to_device(rows)
    d_layers = ctx.alloc(32 * (2 << log_h))
    root = ctx.merkle_commit_rows8(d.ptr, log_h, d_layers.ptr)
    flat = ctx.to_host(d_layers, ((2 << log_h) - 1, 8))
    got, off, k = [], 0, 1 << log_h
    while k >= 1:
        got.append(flat[off:off + k])
        off += k
        k >>= 1
    assert merkle_mismatch(got, exp, mats) is None, merkle_mismatch(got, exp, mats, orc)
    assert root == exp[-1][0].tolist()


# ---------------------------------------------------------------- c. whole segment proofs + query openings
def _segment(width, ncons, nints, seed, quadratic_every=5):
    from powdr_b200 import machine as M
    base = M.synthetic_machine(width, ncons, seed=seed)
    mach = M.SymbolicMachine(base.constraints, M.synthetic_bus(base, nints, seed=seed, quadratic_every=quadratic_every)) if nints else base
    bc, spans = M.compile_constraints(mach)
    return mach, bc, spans, (M.compile_bus(mach, 1) if nints else None)


def _to_monty_host(trace):
    from powdr_b200.capi import R_MOD_P
    return ((trace.astype(np.uint64) * np.uint64(R_MOD_P)) % np.uint64(P)).astype(np.uint32)


def _gpu_segment(ctx, air, trace, log_n, on_device=True):
    width = trace.shape[0]
    if on_device:
        d = ctx.alloc(trace.nbytes).upload(trace)         # canonical words, converted on the device (no 64-bit host copy of a big trace)
        assert ctx.lib.pb_to_monty(ctx.h, C.c_void_p(d.ptr), C.c_size_t(trace.size)) == 0
        proof = ctx.prove_segment(air, d.ptr, log_n, width, on_device=True)
        q, ys = ctx.query_segment(log_n, width, air.perm_width)
        d.free()
    else:
        host = _to_monty_host(trace)
        proof = ctx.prove_segment(air, host.ctypes.data, log_n, width, on_device=False)
        q, ys = ctx.query_segment(log_n, width, air.perm_width)
        del host
    return proof, ys, q


def _cpu_segment(orc, trace, bc, spans, bus, fast, n_queries=8, pow_bits=4):
    return orc.prove(trace, bc, spans, bus, n_queries=n_queries, pow_bits=pow_bits, fast=fast)[:3]


SEGMENTS = {       # log_n, width, constraints, interactions: what each engages
    "2p16_64c_40i": (16, 64, 8, 40),          # smallest fast LDE geometry; the openings reduction over two row splits
    "2p17_300c_300i": (17, 300, 20, 300),     # ~10 generated LogUp modules
    "2p19_160c_60i": (19, 160, 10, 60),       # TMA-staged transposed passes (n_lo = 10)
    "2p20_24c_16i": (20, 24, 4, 16),          # the headline height
    "2p22_4c_2i": (22, 4, 2, 2),              # the (11, 11) pass geometry
}


@pytest.mark.parametrize("name", list(SEGMENTS))
def test_segment_proof_equals_cpu_arm(ctx, orc, monkeypatch, name):
    log_n, width, ncons, nints = SEGMENTS[name]
    fast = _fast(orc, log_n <= 16)
    mach, bc, spans, bus = _segment(width, ncons, nints, seed=log_n)
    trace = rand_field(np.random.default_rng(0xC0FFEE + log_n), (mach.width, 1 << log_n))
    exp = _cpu_segment(orc, trace, bc, spans, bus, fast)
    air = ctx.air(bc, spans, mach.width, bus)
    got = _gpu_segment(ctx, air, trace, log_n)
    assert proof_mismatch(got, exp) is None, "device trace: " + proof_mismatch(got, exp)
    if log_n == 19:
        # the host-input pipeline with 8-column chunks: the ramped schedule (8, 16, 32, ..., 32, 16, 8 + ragged tail) at scale
        monkeypatch.setenv("PB_PIPE_CHUNK_COLS", "8")
        got = _gpu_segment(ctx, air, trace, log_n, on_device=False)
        assert proof_mismatch(got, exp) is None, "host trace, 8-column chunks: " + proof_mismatch(got, exp)
    air.free()


def test_keccak_shape_proof_equals_cpu_arm(ctx, orc):
    """the bench workload: 2^20 rows x 2022 columns, 187 constraints, default FRI parameters (100 queries, 16 PoW bits)"""
    _fast(orc, False)
    log_n, width = 20, 2022
    mach, bc, spans, _ = _segment(width, 187, 0, seed=0xB2000001)
    trace = rand_field(np.random.default_rng(0xB2000001), (width, 1 << log_n))
    exp = _cpu_segment(orc, trace, bc, spans, None, True, n_queries=100, pow_bits=16)
    air = ctx.air(bc, spans, width)
    ctx.set_fri_params(100, 16)
    try:
        got = _gpu_segment(ctx, air, trace, log_n)
    finally:
        ctx.set_fri_params(8, 4)
    del trace
    air.free()
    assert got[0]["n_queries"] == 100 and got[0]["pow_bits"] == 16
    assert proof_mismatch(got, exp) is None, proof_mismatch(got, exp)


def test_headline_bus_proof_equals_cpu_arm(ctx, orc):
    """the 1734-interaction bus of the bench workload (836 chunks, 53 generated LogUp modules) at 2^18 rows"""
    from powdr_b200 import machine as M
    _fast(orc, False)
    log_n = 18
    mach = M.SymbolicMachine([], M.synthetic_bus(2022, 1734, seed=0xB2000002))
    bus = M.compile_bus(mach, 1)
    trace = rand_field(np.random.default_rng(0xB2000002), (mach.width, 1 << log_n))
    exp = _cpu_segment(orc, trace, [], [], bus, True)
    air = ctx.air([], [], mach.width, bus)
    assert air.perm_width == exp[0]["perm_width"] >= 4 * (800 + 1)
    got = _gpu_segment(ctx, air, trace, log_n)
    air.free()
    assert proof_mismatch(got, exp) is None, proof_mismatch(got, exp)


# ---------------------------------------------------------------- d. tuning knobs change the schedule, never the proof
KNOB_SETS = {
    "group1": {"PB_LOGUP_GROUP": "1"}, "group3": {"PB_LOGUP_GROUP": "3"}, "group8": {"PB_LOGUP_GROUP": "8"},
    "perm8_fold4": {"PB_LOGUP_GROUP_PERM": "8", "PB_LOGUP_GROUP_FOLD": "4"},
    "jit_chunks1": {"PB_LOGUP_JIT_CHUNKS": "1"}, "jit_chunks5": {"PB_LOGUP_JIT_CHUNKS": "5"},
    "block64": {"PB_LOGUP_BLOCK": "64", "PB_LOGUP_MINB": "0"}, "block256_minb2": {"PB_LOGUP_BLOCK": "256", "PB_LOGUP_MINB": "2"},
    "block128_minb4": {"PB_LOGUP_BLOCK": "128", "PB_LOGUP_MINB": "4"},
    "air_jit_chunk100": {"PB_AIR_JIT_CHUNK": "100"},      # many AIR modules: the fold passes through the scratch buffer
    "air_no_jit": {"PB_AIR_NO_JIT": "1"},                 # the bytecode interpreter inside the whole LogUp prover
}
_knob_ref = {}         # CPU arm proofs shared by the parameter sets of one test


@pytest.mark.parametrize("knob", list(KNOB_SETS))
def test_tuning_knobs_do_not_change_the_proof(ctx, orc, monkeypatch, knob):
    log_n, width, ncons, nints = SEGMENTS["2p16_64c_40i"]
    mach, bc, spans, bus = _segment(width, ncons, nints, seed=log_n)
    trace = rand_field(np.random.default_rng(0xC0FFEE + log_n), (mach.width, 1 << log_n))
    if "knobs" not in _knob_ref:
        _knob_ref["knobs"] = _cpu_segment(orc, trace, bc, spans, bus, _fast(orc, True))
    for k, v in KNOB_SETS[knob].items():          # set before the AIR is compiled: some are read when the kernels are generated
        monkeypatch.setenv(k, v)
    air = ctx.air(bc, spans, mach.width, bus)
    assert air.is_jit == (knob != "air_no_jit")
    got = _gpu_segment(ctx, air, trace, log_n)
    air.free()
    assert proof_mismatch(got, _knob_ref["knobs"]) is None, proof_mismatch(got, _knob_ref["knobs"])


# ---------------------------------------------------------------- e. multi-chip and sharded provers
@pytest.mark.parametrize("spec", [
    [(14, 64, 0, 120), (12, 40, 0, 60), (9, 30, 3, 0, True), (12, 24, 0, 33)],      # test_gpu_chips.py::test_chips_at_scale_verify
    [(17, 40, 6, 30), (16, 24, 0, 20), (16, 12, 4, 0)],
], ids=["at_scale_verify_spec", "2p17_2p16_2p16"])
def test_chips_proof_equals_cpu_arm(ctx, orc, spec):
    from test_gpu_chips import _chips, _gpu_prove
    fast = _fast(orc, True)
    chips = _chips(spec, seed=9)
    proof, cs, ys, q = _gpu_prove(ctx, chips)
    e_proof, e_cs, e_ys, e_q = orc.prove_chips(chips, n_queries=8, pow_bits=4, fast=fast)
    assert proof_mismatch((proof, ys, q), (e_proof, e_ys, e_q)) is None, proof_mismatch((proof, ys, q), (e_proof, e_ys, e_q))
    assert (cs == e_cs).all(), "cumulative sums: chips %s differ" % np.argwhere((cs != e_cs).any(axis=1)).ravel().tolist()


@pytest.mark.parametrize("on_device", [True, False], ids=["device_trace", "host_trace"])
@pytest.mark.parametrize("world", [2, 4])
def test_sharded_proof_and_queries_equal_cpu_arm(orc, world, on_device):
    from powdr_b200.sharded import prove_segment_threads
    log_n = 17
    mach, bc, spans, bus = _segment(48, 6, 60, seed=log_n + 100)
    trace = rand_field(np.random.default_rng(0x5A4D + log_n), (mach.width, 1 << log_n))
    key = ("sharded", log_n)
    if key not in _knob_ref:
        _knob_ref[key] = _cpu_segment(orc, trace, bc, spans, bus, _fast(orc, True))
    exp = _knob_ref[key]
    for r, (p, q) in enumerate(prove_segment_threads(world, trace, bc, spans, bus=bus, want_queries=True, on_device=on_device)):
        bad = proof_mismatch((p, exp[1], q), exp)
        assert bad is None, "rank %d: %s" % (r, bad)
