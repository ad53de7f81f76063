"""zkml MLP prover: CPU oracle self-checks (-m "not gpu") and GPU-vs-oracle proof parity (-m gpu).
The oracle's zk_prove throws if any of the reference's own invariants fails (dense sumcheck claim,
requant recombination == input evaluation, model-input claim, LogUp fraction cancellation,
final oracle == encode(final_message)); see oracle/zkml.hpp."""
import numpy as np
import pytest
import oracle_py as O


def test_oracle_prover_invariants_hold():
    for nl, w in [(1, 16), (2, 32)]:
        flat, _ = O.zkml_prove(nl, w, 1, 2)
        assert flat.size > 1000
    # different inputs -> different proofs, same input -> same proof (deterministic Fiat-Shamir)
    a, _ = O.zkml_prove(1, 16, 1, 2)
    b, _ = O.zkml_prove(1, 16, 1, 2)
    c, _ = O.zkml_prove(1, 16, 1, 3)
    assert (a == b).all() and (a.size != c.size or not (a == c).all())


def test_synthetic_model_shapes():
    w, b, rq = O.synthetic_mlp(2, 32, 7)
    assert w.min() >= -127 and w.max() <= 127 and b.min() >= -127 and b.max() <= 127
    # requant.rs:395-410: shift is a multiple of BIT_LEN and intermediate_bit_size + fp_scale <= 63
    for r in rq:
        assert (r[0] + r[1]) % 8 == 0 and r[3] + r[1] <= 63


@pytest.mark.gpu
@pytest.mark.parametrize("nl,width", [(1, 16), (2, 32), (2, 256), (3, 512)])
def test_proof_parity(gpu, nl, width):
    """whole proof (all layer proofs, table proofs, commitments, batch opening) bit-exact vs the oracle"""
    w, b, rq = O.synthetic_mlp(nl, width, 11)
    x = O.synthetic_input(width, 12)
    exp, _ = O.zkml_prove(nl, width, 11, 12)
    ctx = gpu.ZkmlContext(nl, width, w, b, rq)
    got = ctx.prove(x)
    if got.shape != exp.shape or not (got == exp).all():
        n = min(got.size, exp.size)
        bad = np.nonzero(got[:n] != exp[:n])[0]
        raise AssertionError("proof differs: sizes %d vs %d, first mismatch at word %s" % (got.size, exp.size, bad[:1]))
    # proving the stored trace gives the same proof (the timed entry point of bench.py)
    ctx.run_inference(x)
    again = ctx.prove_trace(want_proof=True)
    assert (again == exp).all()
    # the concurrent path (bench.py's timed path) keeps the proof of its last job, from the stored trace and end to end
    for e2e in (False, True):
        ctx.prove_concurrent(3, 5, e2e=e2e)
        assert (ctx.last_concurrent_proof() == exp).all()
