import numpy as np

P = 2013265921


def rand_field(rng, shape):
    return rng.integers(0, P, size=shape, dtype=np.uint32)


def bitrev(x, bits):
    r = 0
    for i in range(bits):
        r = (r << 1) | ((x >> i) & 1)
    return r


def bitrev_perm(n_bits):
    return np.array([bitrev(i, n_bits) for i in range(1 << n_bits)], dtype=np.int64)


def root_of_unity(log_n):
    return pow(31, (P - 1) >> log_n, P)


def structured_columns(rng, n, width):
    """`width` columns of height n, the first six the inputs where transform kernels go wrong: all 0, all p-1, alternating
    0 / p-1, a single non-zero at row 0, a single non-zero at row n-1, the ramp i; random columns after them"""
    t = rand_field(rng, (width, n))
    special = [np.zeros(n, np.uint32), np.full(n, P - 1, np.uint32), np.where(np.arange(n) % 2, P - 1, 0).astype(np.uint32),
               np.zeros(n, np.uint32), np.zeros(n, np.uint32), np.arange(n, dtype=np.uint32)]
    special[3][0] = 1 + int(rng.integers(0, P - 1))
    special[4][n - 1] = 1 + int(rng.integers(0, P - 1))
    for c in range(min(width, len(special))):
        t[c] = special[c]
    return t


# ---- first point of divergence, for readable failures at sizes where a whole-array diff is useless ----
def lde_mismatch(got, exp, trace, log_blowup, shift, orc=None):
    """None when equal; else '(column, coset, row)' of the first differing element of two (width, N << log_blowup) LDEs (rows
    bit-reversed), with the scalar oracle's value of that element (the trace polynomial evaluated at the point) when orc is given"""
    if got.shape == exp.shape and np.array_equal(got, exp):
        return None
    if got.shape != exp.shape:
        return "shape %s != %s" % (got.shape, exp.shape)
    bad = np.argwhere(got != exp)
    col, r = int(bad[0][0]), int(bad[0][1])
    n = trace.shape[1]
    log_m = (n << log_blowup).bit_length() - 1
    i_nat = bitrev(r, log_m)
    coset, k = i_nat & ((1 << log_blowup) - 1), i_nat >> log_blowup
    msg = "%d differing elements; first at column %d, coset %d, row %d of the coset (LDE row %d): got %d, expected %d" % (
        len(bad), col, coset, k, r, got[col, r], exp[col, r])
    if orc is not None:
        x = shift * pow(root_of_unity(log_m), i_nat, P) % P
        v = int(orc.eval_at_point(trace[col:col + 1], 1, [x, 0, 0, 0])[0, 0])
        msg += "; scalar oracle says %d (%s is wrong)" % (v, "the kernel" if v == exp[col, r] else "the reference" if v == got[col, r] else "each side")
    return msg


def merkle_mismatch(got, exp, mats, orc=None):
    """got, exp: lists of digest layers (leaves first).  None when equal; else the first differing (layer, node) from the leaves
    up, with the scalar oracle's recomputation of that node from the reference's layer below"""
    for lv, (g, e) in enumerate(zip(got, exp)):
        if np.array_equal(g, e):
            continue
        i = int(np.argwhere((g != e).any(axis=1))[0][0])
        msg = "layer %d (%d nodes): first differing node %d" % (lv, len(e), i)
        if orc is not None:
            if lv == 0:
                v = orc.hash_row(np.concatenate([np.asarray(m)[:, i] for m in mats]))
            else:
                v = orc.compress(exp[lv - 1][2 * i], exp[lv - 1][2 * i + 1])
            msg += "; scalar oracle %s the reference" % ("agrees with" if (v == e[i]).all() else "DISAGREES with")
        return msg
    return None if len(got) == len(exp) else "%d layers != %d" % (len(got), len(exp))


PROOF_ORDER = ("trace_root", "main_root", "logup_alpha", "logup_beta", "perm_root", "cumulative_sum", "alpha", "quotient_root", "zeta",
               "ys", "gamma", "fri_roots", "fri_betas", "final_poly", "pow_witness", "queries")


def proof_mismatch(got, exp):
    """got, exp: (proof dict, ys, queries[, extra arrays by name]).  None when equal; else the first differing item in transcript
    order (roots and challenges, opened values by first index, FRI layers by first index, query openings by first row and word)"""
    (gp, gys, gq), (ep, eys, eq) = got[:3], exp[:3]
    for k in PROOF_ORDER:
        if k == "ys":
            if gys.shape != eys.shape or not np.array_equal(gys, eys):
                if gys.shape != eys.shape:
                    return "opened values: shape %s != %s" % (gys.shape, eys.shape)
                return "opened values: first differing index %d of %d" % (int(np.argwhere((gys != eys).any(axis=1))[0][0]), len(eys))
        elif k == "queries":
            if gq.shape != eq.shape:
                return "query openings: shape %s != %s" % (gq.shape, eq.shape)
            if not np.array_equal(gq, eq):
                q, w = (int(x) for x in np.argwhere(gq != eq)[0])
                return "query openings: first difference at query %d, word %d (opened row index %d)" % (q, w, int(eq[q, 0]))
        elif k in ep or k in gp:
            a, b = gp.get(k), ep.get(k)
            if a != b:
                if isinstance(b, list) and b and isinstance(b[0], list) and isinstance(a, list):
                    i = next((i for i, (x, y) in enumerate(zip(a, b)) if x != y), min(len(a), len(b)))
                    return "%s: first differing entry %d of %d" % (k, i, len(b))
                return "%s: got %s, expected %s" % (k, a, b)
    rest = sorted(k for k in set(gp) | set(ep) if gp.get(k) != ep.get(k))
    return "proof fields %s differ" % rest if rest else None
