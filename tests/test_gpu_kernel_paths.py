"""Each kernel variant the host can select, tested directly against the oracle at the shapes that select it.

The whole-proof tests reach many of these variants only at the shapes their synthetic models happen to produce, and
report a mismatch as "proof differs at word N".  Here every case is named after the path it targets, compares output for
output (every round message, every final evaluation, every layer), and checks through the kernel profile or the launch
counter that the targeted kernel really ran:

- sumcheck rounds: k_sc_lean<2, Base / Ext / Base->Ext / Ext->Ext>, multi-block k_sc_round<1/4/5>, the resident tail
  k_sc_res (1, 2 and 4 CTAs, the warp gather, DSEL 1-5, konst and split bodies, shared operands, its capacity limits),
  each with the resident tail off and on, and at extreme field values (tests/test_oracle_extremes.py crafts inputs that
  take each branch of the accumulators' single reduction);
- MLE primitives: dp_mle_fix_high_new at the k_fixhigh_dot / k_fixhigh_cols switch and with ny == 1, dp_mle_evaluate_many;
- LogUp-GKR: every layer of the fractional-sum circuit (k_logup_den, k_lift_b2e, k_logup_layer, k_logup_tail) and
  dp_mle_linear_combination."""
import ctypes as C
import numpy as np
import pytest
import oracle_py as O
from test_oracle_extremes import CRAFTED_BASE, logup_expected

pytestmark = pytest.mark.gpu
P = O.P


# ---- bindings of the entry points dpb200 does not wrap -----------------------------------------------------------------
def _lib(gpu):
    L = gpu.lib()
    if not getattr(L, "_kernel_paths_ready", False):
        L.dp_mle_fix_high_new.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p)]
        L.dp_mle_fix_high_new.restype = C.c_int
        L.dp_mle_evaluate_many.argtypes = [C.POINTER(C.c_void_p), C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p]
        L.dp_mle_evaluate_many.restype = C.c_int
        L.dp_mle_linear_combination.argtypes = [C.POINTER(C.c_void_p), C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p)]
        L.dp_mle_linear_combination.restype = C.c_int
        L.dp_logup_build.argtypes = [C.POINTER(C.c_void_p), C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]
        L.dp_logup_build.restype = C.c_int
        L.dp_logup_num_vars.argtypes = [C.c_void_p, C.POINTER(C.c_uint32)]
        L.dp_logup_num_vars.restype = C.c_int
        L.dp_logup_outputs.argtypes = [C.c_void_p, C.c_void_p]
        L.dp_logup_outputs.restype = C.c_int
        L.dp_logup_layer_mles.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p), C.POINTER(C.c_uint32)]
        L.dp_logup_layer_mles.restype = C.c_int
        L.dp_logup_free.argtypes = [C.c_void_p]
        L.dp_logup_free.restype = C.c_int
        L.dp_sc_set_resident_tail.argtypes = [C.c_void_p, C.c_int]
        L.dp_sc_set_resident_tail.restype = C.c_int
        L._kernel_paths_ready = True
    return L


def _handles(mles):
    return (C.c_void_p * len(mles))(*[m.h.value for m in mles])


def _u64(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.uint64))


class Profiled:
    """kernel names (dp_profile_read) of the work inside the block"""

    def __init__(self, gpu):
        self.gpu, self.names = gpu, {}

    def __enter__(self):
        self.gpu.profile_enable(True)
        self.gpu.profile_reset()
        return self

    def __exit__(self, *exc):
        try:
            self.names = self.gpu.profile_read()
        finally:
            self.gpu.profile_enable(False)

    def ran(self, prefix):
        return any(n.startswith(prefix) for n in self.names)


# ---- input fills ---------------------------------------------------------------------------------------------------------
def fill(kind, seed, n, ext):
    """rand: splitmix; max: every limb p - 1; alt: 0 / p - 1 alternating by index; c1max: Ext with c1 = p - 1; zero"""
    if kind in ("rand", "chal", "coef") or (kind == "c1max" and not ext):
        return O.splitmix_e(seed, n) if ext else O.splitmix_f(seed, n)
    if kind == "max":
        return np.full((n, 2) if ext else n, P - 1, dtype=np.uint64)
    if kind == "alt":
        v = np.where(np.arange(n) % 2 == 1, P - 1, 0).astype(np.uint64)
        return np.stack([v, v], axis=1) if ext else v
    if kind == "c1max":
        return np.stack([O.splitmix_f(seed, n), np.full(n, P - 1, dtype=np.uint64)], axis=1)
    if kind in ("zero", "sparse"):
        return np.zeros((n, 2) if ext else n, dtype=np.uint64)
    raise ValueError(kind)


def craft_sparse(mles):
    """Operands 0 and 1 of product 0 (same size, both Base or both Ext) get the crafted sums of test_oracle_extremes at
    chosen pairs, zero elsewhere.  A thread of k_sc_lean<2, Base> sums pairs i and i + npairs/2 (2 pairs per thread, grid
    of npairs/512 blocks of 256), so pair b and pair b + npairs/2 hold (x, y) and (x', y') of branch b in the low element
    (evaluation point 0) and those of branch b + 1 in the high one (point 1).  k_sc_lean<2, Ext> gives each thread one
    pair; x = (x, x'), y = (y', y) makes its c1 limb x y + x' y'."""
    (f, ext), (g, _) = mles[0], mles[1]
    f, g = f.copy(), g.copy()
    npairs = (f.shape[0]) // 2
    cases = [CRAFTED_BASE[b] for b in sorted(CRAFTED_BASE)]
    for b in range(len(cases)):
        for half, off in ((0, 0), (1, 1)):
            x, y, x2, y2 = cases[(b + off) % len(cases)]
            i = 2 * b + half
            if ext:
                f[i] = (x, x2); g[i] = (y2, y)
                f[i + npairs] = (x2, x); g[i + npairs] = (y, y2)
            else:
                f[i] = x; g[i] = y
                f[i + npairs] = x2; g[i + npairs] = y2     # element 2 (b + npairs/2) + half
    return [(f, ext), (g, ext)] + mles[2:]


SPECIAL_CH = [(0, 0), (1, 0), (P - 1, 0), (P - 1, P - 1), (P + 3, 0), (P + 5, P + 7), (2, P - 1)]


def challenges(kind, seed, nv):
    """(what the device is given, the canonical values the oracle is given); non-canonical words must act as their value"""
    if kind != "chal":
        ch = O.splitmix_e(seed, nv)
        return ch, ch
    dev = np.array([SPECIAL_CH[i % len(SPECIAL_CH)] for i in range(nv)], dtype=np.uint64)
    return dev, dev % np.uint64(P)


# ---- sumcheck round-kernel matrix --------------------------------------------------------------------------------------
def vp(spec, products, kind, seed):
    """spec: [(num_vars, is_ext)] per MLE; products: [(coef | None, [idx])]"""
    mles = [(fill(kind, seed + i, 1 << nv, ext), ext) for i, (nv, ext) in enumerate(spec)]
    if kind == "sparse":
        mles = craft_sparse(mles)
    out = []
    for j, (coef, idx) in enumerate(products):
        if kind == "coef":
            coef = (P - 1, P - 1)
        elif coef is None:
            coef = tuple(int(v) for v in O.splitmix_e(seed + 100 + j, 1)[0])
        out.append((coef, idx))
    return mles, out


LEAN_B, LEAN_E = "k_sc_lean(msg, Base)", "k_sc_lean(msg, Ext)"
LEAN_BF, LEAN_EF = "k_sc_lean(fold Base->Ext + msg)", "k_sc_lean(fold Ext + msg)"
ROUND_MSG, ROUND_FOLD, RES = "k_sc_round(msg)", "k_sc_round(fold+msg)", "k_sc_res"


def _cases():
    """name -> (nv, spec, products, kernels that must run with the tail off, with the tail on)"""
    c = {}
    for nv in (13, 16):
        deep = [LEAN_BF, LEAN_EF] if nv >= 14 else []          # folding rounds stay lean while a round has > 2048 pairs
        c["lean2_bb_nu%d" % nv] = (nv, [(nv, False)] * 2 + [(nv - 1, False)] * 2, [(None, [0, 1]), (None, [2, 3])], [LEAN_B] + deep, [LEAN_B, RES] + deep)
        c["lean2_ee_nu%d" % nv] = (nv, [(nv, True)] * 2 + [(nv - 2, True)] * 2, [(None, [0, 1]), (None, [3, 2])], [LEAN_E] + deep[1:], [LEAN_E, RES] + deep[1:])
        c["lean2_be_nu%d" % nv] = (nv, [(nv, False), (nv, True), (nv - 1, True), (nv - 1, False)], [(None, [0, 1]), (None, [2, 3])], [ROUND_MSG, ROUND_FOLD], [ROUND_MSG, RES])
        c["lean2_square_nu%d" % nv] = (nv, [(nv, False), (nv - 2, False)], [(None, [0, 0]), (None, [1, 1])], [LEAN_B] + deep, [LEAN_B, RES] + deep)
    c["round4_multiblock_nu13"] = (13, [(13, True), (13, False), (13, False), (13, True), (12, False)] * 1 + [(12, True)] * 3,
                                   [(None, [0, 1, 2, 3]), (None, [4, 5, 6, 7])], [ROUND_MSG, ROUND_FOLD], [ROUND_MSG, ROUND_FOLD, RES])
    c["round5_multiblock_nu13"] = (13, [(13, True), (13, False), (13, True), (13, False), (13, True)], [(None, [0, 1, 2, 3, 4])],
                                   [ROUND_MSG, ROUND_FOLD], [ROUND_MSG, RES])
    c["round1_two_products_nu12"] = (12, [(12, False), (12, True)], [(None, [0]), (None, [1])], [ROUND_MSG, ROUND_FOLD], [ROUND_MSG, RES])
    # resident tail: ncta = 1, 2, 4, 4 (first resident round of 512, 1024, 2048, 2048 pairs); G >= 32 warp gather at nu >= 12;
    # at nu = 13 the tail starts in round 1, after a multi-block round
    for nv in (10, 11, 12, 13):
        c["res_single_nu%d" % nv] = (nv, [(nv, True), (nv, False), (nv, False)], [(None, [0, 1, 2])], [ROUND_MSG, ROUND_FOLD],
                                     [RES] + ([ROUND_MSG] if nv == 13 else []))
    for d in range(1, 6):                                       # uniform degree: k_sc_res<DSEL = d>
        spec = [(9, k % 2 == 0) for k in range(d)] + [(8, k % 2 == 1) for k in range(d)]
        c["res_dsel%d_nu9" % d] = (9, spec, [(None, list(range(d))), (None, list(range(d, 2 * d)))], [ROUND_MSG], [RES])
    # products of nu and nu - 3: 2^3 multiplicity in the glue, then konst products in the last three rounds
    c["res_mixed_nu_konst_nu10"] = (10, [(10, True), (10, False), (7, True), (7, False), (10, True)],
                                    [(None, [0, 1]), (None, [2, 3]), (None, [0, 4, 1]), (None, [3])], [ROUND_MSG], [RES])
    # one MLE (an eq table) in several products, duplicated operands: the swriter / dup bookkeeping
    c["res_shared_operand_nu11"] = (11, [(11, True), (11, False), (11, True), (8, False)],
                                    [(None, [0, 1, 2]), (None, [0, 1]), (None, [0, 2, 2]), (None, [1, 1, 0]), (None, [3, 3])], [ROUND_MSG], [RES])
    # capacity: 96 MLEs / 48 products take the tail (every MLE referenced, 48 x 32 = 1536 pairs <= 2048); 97 or 49 do not
    c["cap_96mles_48products_nu6"] = (6, [(6, k % 3 == 0) for k in range(96)], [(None, [2 * i, 2 * i + 1]) for i in range(48)], [ROUND_MSG], [RES])
    c["cap_97mles_fallback_nu6"] = (6, [(6, k % 3 == 0) for k in range(97)], [(None, [2 * i, 2 * i + 1]) for i in range(47)] + [(None, [94, 95, 96])],
                                    [ROUND_MSG], [ROUND_MSG, "!" + RES])
    c["cap_49products_fallback_nu6"] = (6, [(6, k % 3 == 0) for k in range(96)], [(None, [2 * i, 2 * i + 1]) for i in range(48)] + [(None, [5, 0])],
                                        [ROUND_MSG], [ROUND_MSG, "!" + RES])
    return c


CASES = _cases()
EXTREME_ON = {   # the extreme-value dimension on a subset of the shapes
    "lean2_bb_nu13": ["max", "alt", "sparse", "chal", "coef"],
    "lean2_ee_nu13": ["max", "alt", "c1max", "sparse", "chal"],
    "lean2_square_nu16": ["max", "alt"],
    "lean2_ee_nu16": ["c1max"],
    "round5_multiblock_nu13": ["max", "c1max", "coef"],
    "res_single_nu12": ["max", "alt", "c1max", "chal"],
    "res_dsel3_nu9": ["max", "c1max", "chal", "coef"],
    "res_mixed_nu_konst_nu10": ["alt", "chal"],
}
PARAMS = [(name, "rand") for name in CASES] + [(name, k) for name, ks in EXTREME_ON.items() for k in ks]


def run_sumcheck(gpu, mles, products, nv, ch_dev, ch_ref, tail):
    L = _lib(gpu)
    exp_msgs, exp_fin = O.sumcheck_rounds_fixed(mles, products, nv, ch_ref)
    dm = [gpu.Mle.upload(a, e) for a, e in mles]
    max_deg = max(len(p[1]) for p in products)
    with Profiled(gpu) as prof:
        sc = gpu.Sumcheck(dm, products, nv, max_deg)
        try:
            gpu.check(L.dp_sc_set_resident_tail(sc.h, tail))
            for i in range(nv):
                got = sc.round(None if i == 0 else ch_dev[i - 1])
                assert (got == exp_msgs[i]).all(), "tail=%d round %d: %s != %s" % (tail, i, got.tolist(), exp_msgs[i].tolist())
            assert (sc.finish(ch_dev[nv - 1]) == exp_fin).all(), "tail=%d final evaluations" % tail
        finally:
            sc.destroy()                                     # releases a resident kernel still waiting for a challenge
    for m, (a, ext) in zip(dm, mles):
        assert (m.download().reshape(-1) == a.reshape(-1)).all(), "an input MLE was modified"
    return prof


@pytest.mark.parametrize("name,kind", PARAMS)
def test_sumcheck_round_kernels(gpu, name, kind):
    """every round message and the final evaluations == oracle, with the resident tail off and on; the targeted kernels ran"""
    nv, spec, products, want_off, want_on = CASES[name]
    seed = 7000 + 31 * sum(map(ord, name)) + len(kind)
    mles, prods = vp(spec, products, kind, seed)
    ch_dev, ch_ref = challenges(kind, seed + 1, nv)
    for tail, want in ((0, want_off), (1, want_on)):
        prof = run_sumcheck(gpu, mles, prods, nv, ch_dev, ch_ref, tail)
        for k in want:
            if k.startswith("!"):
                assert not prof.ran(k[1:]), "tail=%d: %s ran (%s)" % (tail, k[1:], sorted(prof.names))
            else:
                assert prof.ran(k), "tail=%d: %s did not run (%s)" % (tail, k, sorted(prof.names))
        if tail == 0:
            assert not prof.ran(RES)


# ---- MLE primitives ------------------------------------------------------------------------------------------------------
def fix_high_new(gpu, m, pt):
    L = _lib(gpu)
    p = _u64(pt).reshape(-1)
    h = C.c_void_p()
    gpu.check(L.dp_mle_fix_high_new(m.h, p.ctypes.data if p.size else None, p.size // 2, C.byref(h)))
    return gpu.Mle(h.value)


# (nv, k, ext) -> launches: eq table (one k_eq_small for k <= 12) + k_fixhigh_dot | k_fixhigh_cols (+ k_sum_parts when ny > 1)
FIX_HIGH_SHAPES = {(9, 5, False): ("k_fixhigh_dot", 2), (10, 5, True): ("k_fixhigh_cols", 3),
                   (19, 1, False): ("k_fixhigh_cols", 2), (20, 2, True): ("k_fixhigh_cols", 2)}


@pytest.mark.parametrize("nv,k,ext", sorted(FIX_HIGH_SHAPES))
@pytest.mark.parametrize("kind", ["rand", "max"])
def test_fix_high_new_switch_points(gpu, nv, k, ext, kind):
    """S = 16 | 32 (k_fixhigh_dot | k_fixhigh_cols) and S = 2^18 (one row band: k_fixhigh_cols writes the output directly,
    no k_sum_parts); the source is left unchanged"""
    f = fill(kind, nv * 7 + k, 1 << nv, ext)
    pt = O.splitmix_e(300 + k, k) if kind == "rand" else np.full((k, 2), P - 1, dtype=np.uint64)
    m = gpu.Mle.upload(f, ext)
    kernel, launches = FIX_HIGH_SHAPES[(nv, k, ext)]
    with Profiled(gpu) as prof:
        before = gpu.lib().dp_kernel_launches()
        r = fix_high_new(gpu, m, pt)
        assert gpu.lib().dp_kernel_launches() - before == launches
        got = r.download()
    assert prof.ran(kernel)
    assert (got == O.fix_high(f, ext, pt)).all()
    assert (m.download() == f).all() and m.info() == (1 << nv, ext, nv)
    assert r.info() == (1 << (nv - k), True, nv - k)


@pytest.mark.parametrize("ext", [False, True])
def test_fix_high_new_k0_is_a_clone(gpu, ext):
    f = fill("rand", 91, 1 << 6, ext)
    m = gpu.Mle.upload(f, ext)
    r = fix_high_new(gpu, m, np.zeros((0, 2), dtype=np.uint64))
    assert r.h.value != m.h.value and gpu.lib().dp_mle_device_ptr(r.h) != gpu.lib().dp_mle_device_ptr(m.h)
    assert r.info() == m.info() and (r.download() == f).all()
    m.free()
    assert (r.download() == f).all()


def evaluate_many(gpu, mles, pt, nv):
    L = _lib(gpu)
    p = _u64(pt).reshape(-1)
    out = np.zeros((len(mles), 2), dtype=np.uint64)
    gpu.check(L.dp_mle_evaluate_many(_handles(mles), len(mles), p.ctypes.data if p.size else None, nv, out.ctypes.data))
    return out


@pytest.mark.parametrize("n,nv", [(1, 13), (16, 12), (17, 0), (17, 1), (17, 12), (17, 13), (17, 16), (17, 17), (40, 16)])
def test_evaluate_many(gpu, n, nv):
    """batches of 16 in k_eval_many (num_vars 1..16), one by one for num_vars 0 and > 16; Base and Ext mixed in one call"""
    srcs = [(fill("max" if i % 5 == 4 else "rand", 500 + i, 1 << nv, i % 2 == 1), i % 2 == 1) for i in range(n)]
    pt = O.splitmix_e(800 + nv, nv) if nv else np.zeros((0, 2), dtype=np.uint64)
    ms = [gpu.Mle.upload(a, e) for a, e in srcs]
    got = evaluate_many(gpu, ms, pt, nv)
    for i, (a, e) in enumerate(srcs):
        exp = O.evaluate(a, e, pt)
        assert (got[i] == exp).all(), "MLE %d" % i
        assert (ms[i].evaluate(pt) == exp).all(), "dp_mle_evaluate, MLE %d" % i


def test_evaluate_many_rejects_mismatched_sizes(gpu):
    ms = [gpu.Mle.upload(O.splitmix_f(1, 16), False), gpu.Mle.upload(O.splitmix_f(2, 8), False)]
    with pytest.raises(gpu.DpError) as e:
        evaluate_many(gpu, ms, O.splitmix_e(3, 4), 4)
    assert e.value.code == gpu.DP_ERR_INVALID


# ---- LogUp circuit -------------------------------------------------------------------------------------------------------
class LogUp:
    def __init__(self, gpu, cols, mults, c, sep):
        self.gpu, self.L = gpu, _lib(gpu)
        self.cols = [gpu.Mle.upload(col, False) for col in cols]
        self.mult = gpu.Mle.upload(mults, False) if mults is not None else None
        cc, ss = _u64(c), _u64(sep)
        self.h = C.c_void_p()
        gpu.check(self.L.dp_logup_build(_handles(self.cols), len(self.cols), self.mult.h if self.mult else None, cc.ctypes.data,
                                        ss.ctypes.data, C.byref(self.h)))

    def num_vars(self):
        v = C.c_uint32()
        self.gpu.check(self.L.dp_logup_num_vars(self.h, C.byref(v)))
        return v.value

    def outputs(self):
        out = np.zeros(8, dtype=np.uint64)
        self.gpu.check(self.L.dp_logup_outputs(self.h, out.ctypes.data))
        return out.reshape(4, 2)

    def layer(self, layer_vars):
        views = (C.c_void_p * 4)()
        n = C.c_uint32()
        self.gpu.check(self.L.dp_logup_layer_mles(self.h, layer_vars, views, C.byref(n)))
        return [self.gpu.Mle(views[i]).download() for i in range(n.value)]

    def free(self):
        if self.h:
            self.L.dp_logup_free(self.h)
            self.h = C.c_void_p()


LOGUP = [  # (len, n_columns, table, fill)
    (4, 1, False, "rand"), (4, 2, True, "rand"), (8, 3, False, "rand"), (8, 16, True, "max"),
    (2048, 2, False, "rand"), (2048, 1, True, "zero-den"), (4096, 3, True, "rand"), (4096, 16, False, "max"),
    (1 << 13, 1, False, "zero-den"), (1 << 13, 2, True, "max"), (1 << 20, 3, False, "rand"), (1 << 20, 2, True, "rand"),
]


@pytest.mark.parametrize("n,ncols,table,kind", LOGUP)
def test_logup_circuit_layers(gpu, n, ncols, table, kind):
    """every layer (through dp_logup_layer_mles views), the outputs and num_vars == the layers built with the oracle's
    arithmetic.  len 2048: the single-block tail from layer 0; 4096: one streaming layer then the tail; larger: several
    streaming layers with grid-stride loops.  zero-den: the constant challenge makes den_0[3] = 0, which must propagate."""
    nv = n.bit_length() - 1
    cols = [fill("max" if kind == "max" else "rand", 40 + k, n, False) for k in range(ncols)]
    mults = O.splitmix_f(60 + n, n) if table else None
    sep = (P - 1, P - 1) if kind == "max" else tuple(int(v) for v in O.splitmix_e(61, 1)[0])
    if kind == "zero-den":
        c = (int(O.f_binop(1, [0], [int(cols[0][3])])[0]), 0)
        if ncols > 1:
            cols[1][3] = 0
    else:
        c = tuple(int(v) for v in O.splitmix_e(62 + n, 1)[0])
    exp = logup_expected(cols, mults, c, sep)
    with Profiled(gpu) as prof:
        lc = LogUp(gpu, cols, mults, c, sep)
        outs = lc.outputs()
    assert prof.ran("k_logup_den") and prof.ran("k_logup_tail")
    assert prof.ran("k_logup_layer") == (n > 2048)
    assert lc.num_vars() == nv - 1
    en, ed = exp[-1]
    assert (outs == np.concatenate([en, ed])).all()
    for layer_vars in range(nv):
        k = nv - 1 - layer_vars
        num, den = exp[k]
        h = 1 << layer_vars
        views = lc.layer(layer_vars)
        want = ([] if (k == 0 and not table) else [num[:h], num[h:]]) + [den[:h], den[h:]]
        assert len(views) == len(want), "layer_vars %d" % layer_vars
        for v, w in zip(views, want):
            assert (v == w).all(), "layer_vars %d" % layer_vars
    if kind == "zero-den":
        assert (exp[0][1][3] == 0).all() and (outs[2 + 1] == 0).all()
    lc.free()


def test_logup_rejects_bad_columns(gpu):
    L = _lib(gpu)
    c = _u64([1, 2])
    h = C.c_void_p()
    cols = [gpu.Mle.upload(O.splitmix_f(k, 16), False) for k in range(17)]
    assert L.dp_logup_build(_handles(cols), 17, None, c.ctypes.data, c.ctypes.data, C.byref(h)) == gpu.DP_ERR_INVALID
    short = [cols[0], gpu.Mle.upload(O.splitmix_f(99, 8), False)]
    assert L.dp_logup_build(_handles(short), 2, None, c.ctypes.data, c.ctypes.data, C.byref(h)) == gpu.DP_ERR_INVALID
    ext = [cols[0], gpu.Mle.upload(O.splitmix_e(98, 16), True)]
    assert L.dp_logup_build(_handles(ext), 2, None, c.ctypes.data, c.ctypes.data, C.byref(h)) == gpu.DP_ERR_INVALID
    bad_mult = gpu.Mle.upload(O.splitmix_f(97, 8), False)
    assert L.dp_logup_build(_handles(cols[:1]), 1, bad_mult.h, c.ctypes.data, c.ctypes.data, C.byref(h)) == gpu.DP_ERR_INVALID


# ---- linear combination ------------------------------------------------------------------------------------------------
def lincomb(gpu, mles, coefs):
    L = _lib(gpu)
    cf = _u64(coefs).reshape(-1)
    h = C.c_void_p()
    gpu.check(L.dp_mle_linear_combination(_handles(mles), cf.ctypes.data, len(mles), C.byref(h)))
    return gpu.Mle(h.value)


@pytest.mark.parametrize("n", [1, 2, 16])
@pytest.mark.parametrize("ln", [1, 1 << 10, 1 << 20])
def test_linear_combination(gpu, n, ln):
    srcs = [fill("max" if k % 4 == 3 else "rand", 200 + k, ln, True) for k in range(n)]
    coefs = O.splitmix_e(400 + n, n)
    coefs[0] = (0, 0)
    if n > 1:
        coefs[1] = (P - 1, P - 1)
    if n > 2:
        coefs[2] = (P - 1, 0)
    exp = np.zeros((ln, 2), dtype=np.uint64)
    for k in range(n):
        exp = O.e_binop(0, exp, O.e_binop(2, np.tile(coefs[k], (ln, 1)), srcs[k]))
    ms = [gpu.Mle.upload(s, True) for s in srcs]
    got = lincomb(gpu, ms, coefs)
    assert got.info() == (ln, True, ln.bit_length() - 1)
    assert (got.download() == exp).all()


def test_linear_combination_rejects(gpu):
    L = _lib(gpu)
    h = C.c_void_p()
    ms = [gpu.Mle.upload(O.splitmix_e(k, 16), True) for k in range(17)]
    cf = _u64(O.splitmix_e(5, 17))
    assert L.dp_mle_linear_combination(_handles(ms), cf.ctypes.data, 17, C.byref(h)) == gpu.DP_ERR_INVALID
    mixed = [ms[0], gpu.Mle.upload(O.splitmix_e(20, 8), True)]
    assert L.dp_mle_linear_combination(_handles(mixed), cf.ctypes.data, 2, C.byref(h)) == gpu.DP_ERR_INVALID
    base = [ms[0], gpu.Mle.upload(O.splitmix_f(21, 16), False)]
    assert L.dp_mle_linear_combination(_handles(base), cf.ctypes.data, 2, C.byref(h)) == gpu.DP_ERR_INVALID
