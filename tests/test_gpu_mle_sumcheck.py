"""GPU parity tests (-m gpu): the CUDA path, called through the C ABI, against the oracle on the same
seeded inputs -- bit-exact (integer arithmetic).  Covers K1-K5 of SURVEY.md section 2."""
import numpy as np
import pytest
import oracle_py as O
from test_oracle_core import rand_vp, vp_sum

pytestmark = pytest.mark.gpu
P = O.P


def test_reference_kat_fix_high(gpu):
    """multilinear_extensions/src/test.rs:47-82 through the device path"""
    evals = np.array([13, 97, 11, 101, 7, 103, 5, 107], dtype=np.uint64)
    pt = np.array([[3, 0], [5, 0]], dtype=np.uint64)
    m = gpu.Mle.upload(evals, False).fix_high(pt[1:])
    exp1 = np.array([[P - 17, 0], [127, 0], [P - 19, 0], [131, 0]], dtype=np.uint64)
    assert (m.download() == exp1).all()
    m2 = gpu.Mle.upload(evals, False).fix_high(pt)
    assert (m2.download() == np.array([[P - 23, 0], [139, 0]], dtype=np.uint64)).all()


def test_upload_canonicalises(gpu):
    v = np.array([P, P + 1, 2**64 - 1, 0, 5, P - 1, 7, 8], dtype=np.uint64)
    got = gpu.Mle.upload(v, False).download()
    assert (got == np.array([0, 1, (2**64 - 1) % P, 0, 5, P - 1, 7, 8], dtype=np.uint64)).all()


@pytest.mark.parametrize("nv", [0, 1, 2, 5, 10, 11, 12, 13, 17, 25])
def test_eq_build(gpu, nv):
    r = O.splitmix_e(50 + nv, nv) if nv else np.zeros((0, 2), dtype=np.uint64)
    assert (gpu.Mle.eq(r).download() == O.build_eq(r)).all()


@pytest.mark.parametrize("nv,k,ext", [(3, 1, False), (6, 6, True), (10, 4, False), (12, 12, False), (14, 5, True),
                                      (16, 10, False), (16, 16, True), (20, 10, False), (20, 10, True),
                                      (9, 5, False), (10, 5, True), (19, 1, False), (20, 2, True)])
def test_fix_high(gpu, nv, k, ext):
    f = O.splitmix_e(nv * 31 + k, 1 << nv) if ext else O.splitmix_f(nv * 31 + k, 1 << nv)
    pt = O.splitmix_e(77 + k, k)
    got = gpu.Mle.upload(f, ext).fix_high(pt).download()
    assert (got == O.fix_high(f, ext, pt)).all()


@pytest.mark.parametrize("nv,k,ext", [(1, 1, False), (8, 3, True), (12, 12, False), (15, 2, False)])
def test_fix_low(gpu, nv, k, ext):
    f = O.splitmix_e(nv + k, 1 << nv) if ext else O.splitmix_f(nv + k, 1 << nv)
    pt = O.splitmix_e(5 + k, k)
    got = gpu.Mle.upload(f, ext).fix_low(pt).download()
    assert (got == O.fix_low(f, ext, pt)).all()


@pytest.mark.parametrize("nv,ext", [(0, False), (0, True), (1, False), (7, True), (12, False), (13, False), (18, True), (21, False)])
def test_evaluate(gpu, nv, ext):
    f = O.splitmix_e(nv + 3, 1 << nv) if ext else O.splitmix_f(nv + 3, 1 << nv)
    pt = O.splitmix_e(900 + nv, nv) if nv else np.zeros((0, 2), dtype=np.uint64)
    assert (gpu.Mle.upload(f, ext).evaluate(pt) == O.evaluate(f, ext, pt)).all()


def test_mle_argument_errors(gpu):
    """reference asserts become status codes (mle.rs:564-567, :609-613)"""
    m = gpu.Mle.upload(np.arange(8, dtype=np.uint64), False)
    with pytest.raises(gpu.DpError) as e:
        m.fix_high(O.splitmix_e(1, 4))
    assert e.value.code == gpu.DP_ERR_INVALID and "invalid size of partial point" in str(e.value)
    with pytest.raises(gpu.DpError) as e:
        m.evaluate(O.splitmix_e(1, 2))
    assert "MLE size does not match the point" in str(e.value)
    with pytest.raises(gpu.DpError):
        gpu.Mle.upload(np.arange(6, dtype=np.uint64), False)


SHAPES = [
    (1, [["b"]]),
    (1, [["e", "b"]]),
    (2, [["b", "b"]]),
    (3, [["b", "b", "b"]]),
    (5, [["e", "b"], ["e"]]),
    (6, [["e", "e", "e"], ["b", "e"], ["b"]]),
    (7, [["b", "b", "b", "b", "b"], ["e", "e", "e", "e"]]),
    (9, [["e", "e", "e", "e", "e"]]),
    (12, [["b", "b", "b"]]),
    (13, [["e", "b"]]),
    (14, [["e", "e", "e"]]),
]


def upload_all(gpu, mles):
    return [gpu.Mle.upload(a, ext) for a, ext in mles]


@pytest.mark.parametrize("nv,shape", SHAPES)
def test_sumcheck_rounds_fixed_challenges(gpu, nv, shape):
    """round-by-round parity with injected challenges: every round message and the final evaluations"""
    mles, products = rand_vp(2000 + nv, nv, shape)
    ch = O.splitmix_e(4, nv)
    exp_msgs, exp_fin = O.sumcheck_rounds_fixed(mles, products, nv, ch)
    dm = upload_all(gpu, mles)
    max_deg = max(len(p[1]) for p in products)
    sc = gpu.Sumcheck(dm, products, nv, max_deg)
    for i in range(nv):
        got = sc.round(None if i == 0 else ch[i - 1])
        assert (got == exp_msgs[i]).all(), "round %d" % i
    assert (sc.finish(ch[nv - 1]) == exp_fin).all()
    # inputs are borrowed, never modified
    for m, (a, ext) in zip(dm, mles):
        assert (m.download().reshape(-1) == a.reshape(-1)).all()


def test_sumcheck_shared_mle_and_mixed_sizes(gpu):
    """eq shared by several products (folded once, virtual_poly.rs:168-177) + smaller-num_vars products
    (2^k multiplicity, sumcheck_macro/src/lib.rs:242-247) + an MLE squared"""
    nv = 8
    eq = (O.build_eq(O.splitmix_e(9, nv)), True)
    a = (O.splitmix_f(1, 1 << nv), False)
    b = (O.splitmix_e(2, 1 << nv), True)
    s1 = (O.splitmix_f(3, 1 << 3), False)
    s2 = (O.splitmix_e(4, 1 << 3), True)
    mles = [eq, a, b, s1, s2]
    products = [((1, 0), [0, 1, 2]), ((7, 3), [0, 1]), ((2, 2), [3, 4]), ((5, 0), [0, 2, 2]), ((1, 1), [3])]
    ch = O.splitmix_e(8, nv)
    exp_msgs, exp_fin = O.sumcheck_rounds_fixed(mles, products, nv, ch)
    sc = gpu.Sumcheck(upload_all(gpu, mles), products, nv, 3)
    for i in range(nv):
        assert (sc.round(None if i == 0 else ch[i - 1]) == exp_msgs[i]).all(), "round %d" % i
    assert (sc.finish(ch[nv - 1]) == exp_fin).all()


@pytest.mark.parametrize("nv,shape", [(4, [["e", "b"], ["b"]]), (10, [["b", "b", "b"]]), (11, [["e", "e"], ["e", "b", "b"]])])
def test_prove_parallel_with_host_fiat_shamir(gpu, nv, shape):
    """IOPProverState::prove_parallel through the C++ host mirror == oracle prove (same Poseidon2 FS),
    and the oracle verifier accepts it"""
    mles, products = rand_vp(3000 + nv, nv, shape)
    point, msgs, fin = gpu.sumcheck_prove_parallel(upload_all(gpu, mles), products, nv)
    opoint, omsgs, ofin = O.sumcheck_prove(mles, products, nv)
    assert (point == opoint).all() and (msgs == omsgs).all() and (fin == ofin).all()
    s = vp_sum(mles, products, nv) if nv <= 10 else O.pe_add(msgs[0][0], msgs[0][1])
    vpoint, _ = O.sumcheck_verify(np.array(s, dtype=np.uint64), nv, max(len(p[1]) for p in products), msgs)
    assert (vpoint == point).all()


def test_sumcheck_full_size_properties(gpu):
    """BASELINE cfg-1 size (nu=20, degree 3, three Base MLEs, splitmix64 seeds 1,2,3): the oracle is too
    slow for an element-wise check in the default suite, so check the size-independent identities of
    sumcheck/src/test.rs:23-56: msg(0)+msg(1) chains through the challenges and the final claim equals
    prod f_i(point)."""
    nv = 20
    mles = [(O.splitmix_f(s, 1 << nv), False) for s in (1, 2, 3)]
    products = [((1, 0), [0, 1, 2])]
    dm = upload_all(gpu, mles)
    point, msgs, fin = gpu.sumcheck_prove_parallel(dm, products, nv)
    s = O.pe_add(msgs[0][0], msgs[0][1])
    vpoint, expected = O.sumcheck_verify(np.array(s, dtype=np.uint64), nv, 3, msgs)
    assert (vpoint == point).all()
    prod = (1, 0)
    for i in range(3):
        ev = dm[i].evaluate(point)
        assert (ev == fin[i]).all()
        prod = O.pe_mul(prod, ev)
    assert prod == tuple(int(v) for v in expected)
    # and the first-round message against the oracle (one pass, cheap)
    omsgs, _ = O.sumcheck_rounds_fixed([(m[0][: 1 << 16], False) for m in mles], products, 16, O.splitmix_e(1, 16))
    sc = gpu.Sumcheck([gpu.Mle.upload(m[0][: 1 << 16], False) for m in mles], products, 16, 3)
    assert (sc.round(None) == omsgs[0]).all()


def test_sumcheck_protocol_errors(gpu):
    """prover.rs:636-639,655,657,710 and virtual_poly.rs:143-160 as status codes"""
    a = gpu.Mle.upload(O.splitmix_f(1, 8), False)
    b = gpu.Mle.upload(O.splitmix_f(2, 4), False)
    with pytest.raises(gpu.DpError) as e:
        gpu.Sumcheck([a, b], [((1, 0), [0, 1])], 3, 2)
    assert "same num_vars" in str(e.value)
    with pytest.raises(gpu.DpError) as e:
        gpu.Sumcheck([a], [((1, 0), [0])], 0, 1)
    assert "Attempt to prove a constant" in str(e.value)
    sc = gpu.Sumcheck([a], [((1, 0), [0])], 3, 1)
    with pytest.raises(gpu.DpError) as e:
        sc.round(np.array([1, 2], dtype=np.uint64))
    assert "first round should be prover first" in str(e.value)
    sc.round(None)
    with pytest.raises(gpu.DpError) as e:
        sc.round(None)
    assert "verifier message is empty" in str(e.value)
    c = np.array([3, 4], dtype=np.uint64)
    sc.round(c); sc.round(c)
    with pytest.raises(gpu.DpError) as e:
        sc.round(c)
    assert e.value.code == gpu.DP_ERR_STATE and "Prover is not active" in str(e.value)
    sc.finish(c)


@pytest.mark.parametrize("nv,shape,T", [(6, [["b", "e"]], 2), (9, [["e", "e", "e"], ["b", "e"]], 4), (12, [["b", "b", "b"]], 8)])
def test_prove_batch_polys(gpu, nv, shape, T):
    """a10: devirgo split on device == oracle == prove_parallel on the un-split polynomial"""
    mles, products = rand_vp(5000 + nv, nv, shape)
    dm = upload_all(gpu, mles)
    point, msgs, fin = gpu.sumcheck_prove_batch_polys(T, dm, products, nv)
    opoint, omsgs, ofin = O.sumcheck_prove(mles, products, nv)
    assert (point == opoint).all() and (msgs == omsgs).all() and (fin == ofin).all()


def test_resident_tail_is_released_when_the_prover_is_dropped(gpu):
    """the resident tail kernel (dp_sc_set_resident_tail) waits for challenges on the device; dropping the handle in the
    middle of a proof must release it (abort word) instead of leaving a spinning kernel behind, and the library must keep
    working afterwards.  Also: with and without the tail the round messages are identical."""
    import ctypes as C
    nv = 9
    mles = [(O.splitmix_f(71, 1 << nv), False), (O.splitmix_e(72, 1 << nv), True)]
    products = [((2, 3), [0, 1]), ((1, 0), [1, 1, 0])]
    ch = O.splitmix_e(73, nv)
    exp_msgs, exp_fin = O.sumcheck_rounds_fixed(mles, products, nv, ch)
    for tail in (0, 1):
        sc = gpu.Sumcheck([gpu.Mle.upload(a, e) for a, e in mles], products, nv, 3)
        gpu.check(gpu.lib().dp_sc_set_resident_tail(sc.h, tail))
        got = [sc.round(None)] + [sc.round(ch[i - 1]) for i in range(1, nv)]
        assert (np.array(got) == exp_msgs).all()
        assert (sc.finish(ch[nv - 1]) == exp_fin).all()
        sc.destroy()
    sc = gpu.Sumcheck([gpu.Mle.upload(a, e) for a, e in mles], products, nv, 3)
    gpu.check(gpu.lib().dp_sc_set_resident_tail(sc.h, 1))
    sc.round(None); sc.round(ch[0]); sc.round(ch[1])      # tables are <= 128 pairs from round 2 on: the tail kernel is now waiting
    sc.destroy()                                           # must post the abort word and return
    m = gpu.Mle.upload(mles[0][0], False)
    assert (m.evaluate(ch) == O.evaluate(mles[0][0], False, ch)).all()   # the stream is usable again


def test_final_evaluations_follow_caller_order(gpu):
    """round-1 advisor finding: VirtualPolynomial numbers MLEs by first use (virtual_poly.rs:168-177); the C entry points must report
    final evaluations in the CALLER's order even when the first product references [2, 0] and MLE 1 is referenced by nobody
    (its slot is zero: it is not part of the VirtualPolynomial).  prove_parallel, prove_batch_polys and prove_sharded agree."""
    import multigpu as mg
    nv = 8
    mles = [(O.splitmix_f(1, 1 << nv), False), (O.splitmix_e(2, 1 << nv), True), (O.splitmix_f(3, 1 << nv), False), (O.splitmix_f(4, 1 << nv), False)]
    products = [((1, 0), [2, 0]), ((2, 1), [0, 3, 2])]
    ep, em, ef = O.sumcheck_prove(mles, products, nv)
    exp_fin = ef.copy(); exp_fin[1] = 0
    for name, run in (("parallel", lambda dm: gpu.sumcheck_prove_parallel(dm, products, nv)),
                      ("batch", lambda dm: gpu.sumcheck_prove_batch_polys(4, dm, products, nv)),
                      ("sharded-native", lambda dm: mg.prove_sharded_native(dm, products, nv, 0, 1, allgather=lambda w: w[None, :])),
                      ("sharded-python", lambda dm: mg.prove_sharded_device(dm, products, nv, 0, 1, None))):
        point, msgs, fin = run(upload_all(gpu, mles))
        assert (np.asarray(point) == ep).all() and (np.asarray(msgs) == em).all(), name
        fin = np.asarray(fin)
        for i in (0, 2, 3):
            assert (fin[i] == exp_fin[i]).all(), (name, i)
        if name != "sharded-python":      # the Python path folds every MLE it is given, referenced or not
            assert (fin[1] == 0).all(), name
