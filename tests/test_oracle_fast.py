"""The CPU reference arm (oracle/fast.c: AVX-512 Montgomery) against the scalar `%`-based restatement, bit for bit, on every
primitive it re-implements -- so that timing it (bench.py cpu_baseline / --impl reference) times the same computation."""
import numpy as np
import pytest

from util import P, rand_field, root_of_unity, structured_columns, lde_mismatch, merkle_mismatch, proof_mismatch


@pytest.fixture(scope="module")
def fast(orc):
    if not orc.fast_available():
        pytest.skip("host CPU has no AVX-512")
    return orc


@pytest.mark.parametrize("log_n,width,log_blowup,shift", [(1, 2, 1, 31), (3, 3, 1, 31), (4, 2, 1, 31), (5, 3, 2, 31), (8, 5, 1, 1), (10, 4, 1, 1234567), (13, 3, 1, 31)])
def test_fast_lde(fast, log_n, width, log_blowup, shift):
    rng = np.random.default_rng(log_n)
    t = rand_field(rng, (width, 1 << log_n))
    t[0, :2] = [0, P - 1]
    assert (fast.fast_lde_batch(t, log_blowup, shift) == fast.lde_batch(t, log_blowup, shift)).all()


@pytest.mark.parametrize("widths,log_h", [([3], 2), ([8], 4), ([17], 5), ([8, 8], 6), ([5, 2, 9], 7), ([33], 10)])
def test_fast_merkle(fast, widths, log_h):
    rng = np.random.default_rng(log_h)
    mats = [rand_field(rng, (w, 1 << log_h)) for w in widths]
    a, b = fast.fast_merkle_commit(mats), fast.merkle_commit(mats)
    for x, y in zip(a, b):
        assert (x == y).all()


def test_fast_quotient_and_fold(fast):
    from powdr_b200 import machine as M
    mach = M.synthetic_machine(40, 11, seed=5)
    bc, spans = M.compile_constraints(mach)
    bc = list(bc) + [M.OP_PUSH_APC, 3, M.OP_INV_OR_ZERO, M.OP_PUSH_APC, 4, M.OP_MUL, M.OP_PUSH_CONST, P - 5, M.OP_ADD, M.OP_NEG]
    spans = list(spans) + [(len(bc) - 10, 10)]
    rng = np.random.default_rng(3)
    log_n = 6
    lde = rand_field(rng, (mach.width, 2 << log_n))
    lde[3, :5] = 0
    alpha = rand_field(rng, 4)
    assert (fast.fast_quotient(bc, spans, lde, log_n, alpha) == fast.quotient(bc, spans, lde, log_n, alpha)).all()
    assert (fast.fast_constraint_fold(bc, spans, lde, alpha) == fast.constraint_fold(bc, spans, lde, alpha)).all()


def test_fast_openings_and_reduced_opening(fast):
    rng = np.random.default_rng(4)
    log_n, w = 7, 6
    t = rand_field(rng, (w, 1 << log_n))
    zeta, gamma = rand_field(rng, 4), rand_field(rng, 4)
    for shift in (1, 31, 777):
        assert (fast.fast_eval_at_point(t, shift, zeta) == fast.eval_at_point(t, shift, zeta)).all()
    lde = fast.lde_batch(t, 1, 31)
    other = rand_field(rng, (3, 2 << log_n))
    ys = rand_field(rng, (w + 3, 4))
    assert (fast.fast_deep_quotient([lde, other], 31, zeta, gamma, ys) == fast.deep_quotient([lde, other], 31, zeta, gamma, ys)).all()


# ---- the sizes the CPU arm vouches for when the GPU is checked against it (tests/test_gpu_scale_parity.py): past BLK_LOG = 18 in
# oracle/fast.c, where the cache-blocked NTT stages and the tiled bit reversal take over, and whole proofs at 2^16 ----
def _w2n_inv(log_n):
    return pow(root_of_unity(log_n + 1), P - 2, P)


@pytest.mark.parametrize("log_n,width,log_blowup,shift", [(19, 8, 1, 31), (19, 7, 1, 1), (19, 7, 1, "w2n_inv"), (19, 7, 2, 31), (20, 8, 1, 31),
                                                          (20, 7, 1, "w2n_inv"), (21, 7, 1, 31)])
def test_fast_lde_past_the_blocked_stages(fast, log_n, width, log_blowup, shift):
    shift = _w2n_inv(log_n) if shift == "w2n_inv" else shift
    t = structured_columns(np.random.default_rng(1000 + log_n), 1 << log_n, width)
    got, exp = fast.fast_lde_batch(t, log_blowup, shift), fast.lde_batch(t, log_blowup, shift)
    assert lde_mismatch(got, exp, t, log_blowup, shift) is None, lde_mismatch(got, exp, t, log_blowup, shift, fast)


@pytest.mark.parametrize("widths,log_h", [([4, 4], 17), ([3, 16], 18)])
def test_fast_merkle_every_layer_at_scale(fast, widths, log_h):
    rng = np.random.default_rng(log_h)
    mats = [rand_field(rng, (w, 1 << log_h)) for w in widths]
    got, exp = fast.fast_merkle_commit(mats), fast.merkle_commit(mats)
    assert merkle_mismatch(got, exp, mats) is None, merkle_mismatch(got, exp, mats, fast)


def test_fast_prove_equals_scalar_prove_at_2p16_with_interactions(fast):
    """64 columns, 8 constraints, 40 interactions (a quadratic one every 7th): the proof, the opened values and the query openings"""
    from powdr_b200 import machine as M
    base = M.synthetic_machine(64, 8, seed=16)
    mach = M.SymbolicMachine(base.constraints, M.synthetic_bus(base, 40, seed=16, quadratic_every=7))
    bc, spans = M.compile_constraints(mach)
    bus = M.compile_bus(mach, 1)
    trace = rand_field(np.random.default_rng(16), (mach.width, 1 << 16))
    got, exp = fast.prove(trace, bc, spans, bus, fast=True)[:3], fast.prove(trace, bc, spans, bus)[:3]
    assert proof_mismatch(got, exp) is None, proof_mismatch(got, exp)


def test_fast_prove_chips_equals_scalar_with_a_2p15_chip(fast):
    from test_oracle_chips import _chips
    chips = _chips([(15, 24, 3, 12), (13, 40, 0, 20), (11, 9, 4, 0), (13, 16, 2, 6)], seed=15)
    gp, gcs, gys, gq = fast.prove_chips(chips, fast=True)
    ep, ecs, eys, eq = fast.prove_chips(chips)
    assert proof_mismatch((gp, gys, gq), (ep, eys, eq)) is None, proof_mismatch((gp, gys, gq), (ep, eys, eq))
    assert (gcs == ecs).all()
