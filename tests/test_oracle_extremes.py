"""The oracle against plain Python integers at the extreme field values, and a bit-level model of the device's single
reduction of an unreduced accumulator (gl_reduce128_weak -> gl_reduce160 -> gl_canon_weak, csrc/gl.cuh) used to pick
inputs that drive each of its branches.  CPU only: the GPU parity tests compare the kernels with the oracle, so an error
the two shared would hide there; here the oracle meets arithmetic that cannot share it.

The crafted inputs (CRAFTED_*) and the LogUp layer builder are imported by tests/test_gpu_kernel_paths.py."""
import itertools
import numpy as np
import pytest
import oracle_py as O

P = O.P
M64 = (1 << 64) - 1
EPS = 0xFFFFFFFF


# ---- model of the device reduction ----------------------------------------------------------------------------------
def reduce128_weak(lo, hi):
    """gl_reduce128_weak as its PTX computes it: (weak result in [0, 2^64), borrow taken, carry taken)"""
    hl, hh = hi & EPS, hi >> 32
    t0 = lo - hh
    borrow = t0 < 0
    if borrow:
        t0 = t0 + (1 << 64) - EPS           # 2^96 == -1: the borrow adds p, i.e. subtracts EPS mod 2^64
    assert 0 <= t0 <= M64
    t0 += hl * EPS                          # 2^64 == EPS
    carry = t0 > M64
    r = (t0 & M64) + (EPS if carry else 0)
    assert r <= M64                         # "cannot carry again"
    return r, borrow, carry


def reduce160(lo, hi, top):
    """gl_reduce160 (with its gl_canon_weak): (canonical result, {branch: taken})"""
    assert 0 <= top < 1 << 31
    r, borrow, carry = reduce128_weak(lo, hi)
    d = r - (top << 32)                     # 2^128 == -2^32
    sub_borrow = d < 0
    if sub_borrow:
        d = d + (1 << 64) - EPS
    assert 0 <= d <= M64
    weak = d >= P                           # gl_canon_weak subtracts p
    return (d - P if weak else d), {"borrow": borrow, "carry": carry, "top": top > 0, "sub_borrow": sub_borrow, "weak": weak}


def acc_reduce(total):
    """one acc192 / eacc limb: the exact integer sum of the raw products, reduced once"""
    assert 0 <= total < 1 << 159
    return reduce160(total & M64, (total >> 64) & M64, total >> 128)


def eacc_limbs(terms):
    """k_sc_lean's eacc over the pairs (x, y) of Ext elements one thread multiplies: the integer sums the two limbs reduce
    (c1 = x0 y1 + x1 y0, c0 = x0 y0 + 7 weak(x1 y1))"""
    c0 = c1 = 0
    for (x0, x1), (y0, y1) in terms:
        c1 += x0 * y1 + x1 * y0
        w, _, _ = reduce128_weak((x1 * y1) & M64, (x1 * y1) >> 64)
        c0 += x0 * y0 + 7 * w
    return c0, c1


# ---- structured search for inputs that take each branch ---------------------------------------------------------------
def _family():
    small = [0, 1, 2, 3, 7]
    v = set(small)
    for a in small + [EPS]:
        v.update([P - 1 - a, (1 << 63) + a, (1 << 63) - 1 - a])
        for k in (1, 2, 3, 4, 1 << 16, 1 << 31, EPS - 1, EPS):
            v.update([k * (1 << 32) + a, k * (1 << 32) - 1 - a])
    return sorted(x % P for x in v)


FAMILY = _family()
BRANCHES = ("borrow", "carry", "top", "sub_borrow", "weak")


def search_two_term():
    """two-term sums x*y + x'*y' -- the sums a thread of k_sc_lean<2, Base> forms over its two pairs -- checked against % p:
    x, y over the family with (x', y') in {(p - x, y), (x, y), (y, x), (0, 0)}, and (p - 1)^2 + x' y' with x', y' over the
    family; returns {branch: first (x, y, x', y')}"""
    found = {}
    checked = 0
    cands = [(x, y, x2, y2) for x, y in itertools.product(FAMILY, repeat=2) for x2, y2 in (((P - x) % P, y), (x, y), (y, x), (0, 0))]
    cands += [(P - 1, P - 1, x2, y2) for x2, y2 in itertools.product(FAMILY, repeat=2)]
    for x, y, x2, y2 in cands:
        s = x * y + x2 * y2
        got, br = acc_reduce(s)
        assert got == s % P, (x, y, x2, y2)
        checked += 1
        for b in BRANCHES:
            if br[b] and b not in found:
                found[b] = (x, y, x2, y2)
    return found, checked


_FOUND, _CHECKED = search_two_term()
# (x, y, x', y') per branch: placed by the GPU tests at a thread's two pairs so that ONE accumulator holds exactly x y + x' y'
CRAFTED_BASE = dict(_FOUND)


def test_reduction_model_matches_mod_p_on_the_search():
    assert _CHECKED > 10000
    # every branch of the single reduction is reachable from two canonical products (the sub-borrow needs r < top 2^32 with
    # top > 0, which two products near 2^128 give)
    assert set(CRAFTED_BASE) == set(BRANCHES), "branches without a crafted input: %s" % (set(BRANCHES) - set(CRAFTED_BASE))


def test_reduction_model_edges():
    for lo, hi, top in [(0, 0, 0), (M64, M64, 0), (M64, M64, (1 << 31) - 1), (P, 0, 0), (P - 1, 0, 0), (0, EPS << 32, 0),
                        (EPS - 1, 1 << 32, 0), (0, 0, 1), (M64, 0, 1), (5, EPS, 3)]:
        got, _ = reduce160(lo, hi, top)
        assert got == (lo + (hi << 64) + (top << 128)) % P


def test_crafted_inputs_take_their_branch():
    for b, (x, y, x2, y2) in CRAFTED_BASE.items():
        assert all(0 <= v < P for v in (x, y, x2, y2))
        assert acc_reduce(x * y + x2 * y2)[1][b]


def test_ext_accumulator_limbs_reach_the_carry_and_top_branches():
    """the Ext lean kernels reduce c0 = x0 y0 + 7 weak(x1 y1) and c1 = x0 y1 + x1 y0 once: with c1 = p - 1 operands (the
    GPU tests' "c1max" fill) the 7 w term is largest and both limbs pass 2^128"""
    x = y = (P - 1, P - 1)
    c0, c1 = eacc_limbs([(x, y)])
    assert acc_reduce(c0)[0] == c0 % P and acc_reduce(c1)[0] == c1 % P
    assert acc_reduce(c1)[1]["top"]
    ref = O.pe_mul(x, y)
    assert (c0 % P, c1 % P) == ref


# ---- the oracle's field arithmetic against Python integers -------------------------------------------------------------
EXTREME = [0, 1, 2, 7, EPS, 1 << 32, (1 << 32) + 1, 1 << 63, (1 << 63) + 1, P - (1 << 32), P - 2, P - 1]


def test_oracle_base_ops_at_extremes():
    a = np.array([x for x in EXTREME for _ in EXTREME], dtype=np.uint64)
    b = np.array([y for _ in EXTREME for y in EXTREME], dtype=np.uint64)
    for op, fn in ((0, lambda x, y: (x + y) % P), (1, lambda x, y: (x - y) % P), (2, lambda x, y: x * y % P)):
        got = O.f_binop(op, a, b)
        assert [int(v) for v in got] == [fn(int(x), int(y)) for x, y in zip(a, b)]


def test_oracle_ext_ops_at_extremes():
    vals = [(x, y) for x in (0, 1, P - 1, 1 << 63, EPS) for y in (0, 1, P - 1, (1 << 32) + 1)]
    a = np.array([u for u in vals for _ in vals], dtype=np.uint64)
    b = np.array([v for _ in vals for v in vals], dtype=np.uint64)
    for op, fn in ((0, O.pe_add), (1, O.pe_sub), (2, O.pe_mul)):
        got = O.e_binop(op, a, b)
        assert [tuple(int(v) for v in r) for r in got] == [fn(x, y) for x, y in zip(a, b)]


# ---- MLE primitives of the oracle against Python integers -------------------------------------------------------------
def py_eq(point):
    t = [(1, 0)]
    for r in point:                                   # variable b is bit b of the index (build_eq_x_r_vec)
        one_m = O.pe_sub((1, 0), r)
        t = [O.pe_mul(v, one_m) for v in t] + [O.pe_mul(v, r) for v in t]
    return t


def py_fix_high(ev, point):
    """fix the HIGH len(point) variables: out[i] = sum_j eq(point)[j] ev[j S + i]"""
    w = py_eq(point)
    S = len(ev) >> len(point)
    out = []
    for i in range(S):
        acc = (0, 0)
        for j, wj in enumerate(w):
            acc = O.pe_add(acc, O.pe_mul(wj, ev[j * S + i]))
        out.append(acc)
    return out


def _ext(ev, is_ext):
    return [tuple(int(v) for v in e) for e in ev] if is_ext else [(int(v), 0) for v in ev]


EXT_FILLS = {
    "max": lambda n: np.full((n, 2), P - 1, dtype=np.uint64),
    "alt": lambda n: np.array([[0, 0] if i % 2 else [P - 1, P - 1] for i in range(n)], dtype=np.uint64),
    "c1max": lambda n: np.stack([O.splitmix_f(17, n), np.full(n, P - 1, dtype=np.uint64)], axis=1),
}
PTS = [np.array([[P - 1, P - 1]] * 4, dtype=np.uint64), np.array([[0, 0], [1, 0], [P - 1, 0], [P - 1, P - 1]], dtype=np.uint64)]


@pytest.mark.parametrize("fill", sorted(EXT_FILLS))
@pytest.mark.parametrize("is_ext", [False, True])
def test_oracle_mle_ops_at_extremes(fill, is_ext):
    nv = 4
    ev = EXT_FILLS[fill](1 << nv)
    if not is_ext:
        ev = ev[:, 0].copy()
    pev = _ext(ev, is_ext)
    for pt in PTS:
        ppt = [tuple(int(v) for v in r) for r in pt]
        assert _ext(O.build_eq(pt), True) == py_eq(ppt)
        for k in (1, 3, 4):
            assert _ext(O.fix_high(ev, is_ext, pt[:k]), True) == py_fix_high(pev, ppt[:k])
        assert tuple(int(v) for v in O.evaluate(ev, is_ext, pt)) == py_fix_high(pev, ppt)[0]


# ---- sumcheck rounds of the oracle against Python integers ------------------------------------------------------------
def _lagrange(evals, at):
    n = len(evals)
    res = (0, 0)
    for j in range(n):
        num = den = 1
        for i in range(n):
            if i != j:
                num = num * (at - i) % P
                den = den * (j - i) % P
        res = O.pe_add(res, O.pe_mul(evals[j], (num * pow(den, P - 2, P) % P, 0)))
    return res


def py_sumcheck_rounds(tables, products, nv, ch):
    """the round messages with fixed challenges, every MLE with nv variables: fold the low variable by the previous
    challenge, then sum each product over the pairs at t = 0..deg, extrapolate to max_deg, add up"""
    tabs = [list(t) for t in tables]
    max_deg = max(len(p[1]) for p in products)
    msgs = []
    for r in range(nv):
        if r:
            c = ch[r - 1]
            tabs = [[O.pe_add(t[2 * i], O.pe_mul(O.pe_sub(t[2 * i + 1], t[2 * i]), c)) for i in range(len(t) // 2)] for t in tabs]
        msg = [(0, 0)] * (max_deg + 1)
        for coef, idx in products:
            d = len(idx)
            sums = []
            for t in range(d + 1):
                acc = (0, 0)
                for i in range(len(tabs[idx[0]]) // 2):
                    pr = (1, 0)
                    for m in idx:
                        lo, hi = tabs[m][2 * i], tabs[m][2 * i + 1]
                        pr = O.pe_mul(pr, O.pe_add(lo, O.pe_mul((t, 0), O.pe_sub(hi, lo))))
                    acc = O.pe_add(acc, pr)
                sums.append(O.pe_mul(acc, coef))
            sums += [_lagrange(sums, x) for x in range(d + 1, max_deg + 1)]
            msg = [O.pe_add(a, b) for a, b in zip(msg, sums)]
        msgs.append(msg)
    c = ch[nv - 1]
    fin = [O.pe_add(t[0], O.pe_mul(O.pe_sub(t[1], t[0]), c)) for t in tabs]
    return msgs, fin


@pytest.mark.parametrize("fill", ["max", "alt", "c1max", "rand"])
def test_oracle_sumcheck_rounds_at_extremes(fill):
    nv = 3
    n = 1 << nv
    mk = EXT_FILLS.get(fill, lambda n: O.splitmix_e(5, n))
    mles = [(mk(n), True), (EXT_FILLS["max"](n)[:, 0].copy(), False), (mk(n)[::-1].copy(), True), (O.splitmix_f(9, n), False)]
    products = [((P - 1, P - 1), [0, 1]), ((1, 0), [2, 2, 3]), ((3, P - 1), [0, 1, 2, 3, 0]), ((P - 1, 0), [3])]
    ch = np.array([[P - 1, P - 1], [0, 0], [1, 0]], dtype=np.uint64)
    msgs, fin = O.sumcheck_rounds_fixed(mles, products, nv, ch)
    pmsgs, pfin = py_sumcheck_rounds([_ext(a, e) for a, e in mles], products, nv, [tuple(int(v) for v in c) for c in ch])
    assert [[tuple(int(v) for v in e) for e in m] for m in msgs] == pmsgs
    assert [tuple(int(v) for v in e) for e in fin] == pfin


# ---- LogUp fractional-sum circuit: the expected layers, built with the oracle's arithmetic ---------------------------
def logup_expected(cols, mults, c, sep):
    """layers [(num, den)] of LogUpCircuit::new_{lookup,table}_circuit: den_0 = c + sum_k sep^k col_k, num_0 = -1 (lookup) or
    the lifted multiplicities (table); layer k+1 pairs i with i + half: n = n1 d2 + d1 n2, d = d1 d2"""
    n = cols[0].size
    den = np.tile(np.asarray(c, dtype=np.uint64), (n, 1))
    pw = np.array([[1, 0]], dtype=np.uint64)
    for col in cols:
        lifted = np.stack([col, np.zeros_like(col)], axis=1)
        den = O.e_binop(0, den, O.e_binop(2, np.tile(pw, (n, 1)), lifted))
        pw = O.e_binop(2, pw, np.asarray(sep, dtype=np.uint64).reshape(1, 2))
    if mults is None:
        num = np.tile(np.array([P - 1, 0], dtype=np.uint64), (n, 1))
    else:
        num = np.stack([mults, np.zeros_like(mults)], axis=1)
    layers = [(num, den)]
    while num.shape[0] > 2:
        h = num.shape[0] // 2
        n1, n2, d1, d2 = num[:h], num[h:], den[:h], den[h:]
        num = O.e_binop(0, O.e_binop(2, n1, d2), O.e_binop(2, d1, n2))
        den = O.e_binop(2, d1, d2)
        layers.append((num, den))
    return layers


def logup_expected_py(cols, mults, c, sep):
    n = len(cols[0])
    den = []
    for i in range(n):
        acc, pw = tuple(c), (1, 0)
        for col in cols:
            acc = O.pe_add(acc, O.pe_mul(pw, (int(col[i]), 0)))
            pw = O.pe_mul(pw, tuple(sep))
        den.append(acc)
    num = [(P - 1, 0)] * n if mults is None else [(int(m), 0) for m in mults]
    layers = [(num, den)]
    while len(num) > 2:
        h = len(num) // 2
        num, den = ([O.pe_add(O.pe_mul(num[i], den[i + h]), O.pe_mul(den[i], num[i + h])) for i in range(h)],
                    [O.pe_mul(den[i], den[i + h]) for i in range(h)])
        layers.append((num, den))
    return layers


@pytest.mark.parametrize("n,ncols,table,fill", [(4, 1, False, "rand"), (8, 2, True, "rand"), (16, 3, False, "max"),
                                                (64, 16, True, "max"), (32, 2, False, "zero-den")])
def test_logup_expected_layers_against_python_integers(n, ncols, table, fill):
    cols = [O.splitmix_f(40 + k, n) if fill != "max" else np.full(n, P - 1, dtype=np.uint64) for k in range(ncols)]
    mults = O.splitmix_f(60, n) if table else None
    sep = (P - 1, P - 1) if fill == "max" else tuple(int(v) for v in O.splitmix_e(61, 1)[0])
    c = (int(P - cols[0][3]), 0) if fill == "zero-den" else tuple(int(v) for v in O.splitmix_e(62, 1)[0])
    if fill == "zero-den":
        cols = cols[:1] + [np.zeros(n, dtype=np.uint64)]        # den_0[3] == 0 exactly
    got = logup_expected(cols, mults, c, sep)
    ref = logup_expected_py(cols, mults, c, sep)
    assert len(got) == len(ref) == n.bit_length() - 1
    for (gn, gd), (rn, rd) in zip(got, ref):
        assert _ext(gn, True) == rn and _ext(gd, True) == rd
    if fill == "zero-den":
        assert ref[0][1][3] == (0, 0) and ref[-1][1][3 % 2] == (0, 0)     # the zero follows index 3 mod half down to the output
