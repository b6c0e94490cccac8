"""SuperNova's `compress` on the CPU: the batched Spartan verifier and batch_eval_reduce's verifier (tests/spartan_batched_oracle.py)
against the pure-Python batched prover that follows the same list as the GPU prover (lurk-beta_b200/spartan.py:
BatchedRelaxedR1CSProver).  Accepts 1, 2 and 3 genuinely folded relaxed-R1CS instances of different shapes; rejects a tampered E, a
changed u, swapped instances and a wrong reduced evaluation.  Also: lurk_poly_combine_dev's argument checks (no GPU needed)."""
import numpy as np
import pytest

from oracle import sumcheck as sc
from spartan_batched_oracle import batch_eval_verify, eval_claims, powers, python_batched_prover, shape, verify_batched
from test_gpu_spartan_chain import challenge, folded_instance, rows_of
from util import ints

# (frames, slot_elems, glue, lin_rows): rows = frames (2 glue + lin_rows), n_w = frames (slot_elems + glue)
SHAPES = [(3, 10, 5, 4),       # 42 rows (2^6), 45 variables (z: 2^7)
          (2, 12, 3, 2),       # 16 rows (2^4), 30 variables (z: 2^6)
          (1, 6, 4, 60)]       # 68 rows (2^7), 10 variables (z: 2^5): the most rows, not the most variables


def instance(oracle, spec, seed, shp):
    mats, n_w, o = folded_instance(oracle, spec, np.random.default_rng(seed), *shp)
    return dict(mats=mats, R=[rows_of(m) for m in mats], n_w=n_w, rows=len(mats[0][0]) - 1, W=ints(o.W), E=ints(o.E), u=o.u, X=list(o.X))


@pytest.fixture(scope="module")
def instances(oracle, spec):
    return [instance(oracle, spec, 31 + i, shp) for i, shp in enumerate(SHAPES)]


def check(insts, proof, p):
    """both verifiers; returns the reduced claim (rho, v, gamma powers) or None"""
    ok, rx, ry = verify_batched(insts, proof, challenge, p)
    if not ok:
        return None
    pts = eval_claims(insts, proof, rx, ry)
    b = proof["batch"]
    return batch_eval_verify(b["rounds"], [x for x, _ in pts], [v for _, v in pts], b["left"], challenge, p)


@pytest.mark.parametrize("k", [1, 2, 3])
def test_batched_verifier_accepts_folded_instances(spec, instances, k):
    p = spec.FIELD_MODULUS[0]
    insts = instances[:k]
    if k == 3:
        sh = [shape(I) for I in insts]
        assert max(range(3), key=lambda i: sh[i][0]) != max(range(3), key=lambda i: sh[i][2])   # r_x and r_y suffixes differ
    proof = python_batched_prover(insts, challenge, p)
    got = check(insts, proof, p)
    assert got is not None
    rho, v, gp = got
    b = proof["batch"]
    assert rho == b["rho"] and v == b["v"] and gp == powers(b["gamma"], 2 * k, p)
    # the one opening: the joint polynomial (zero-extended claims) evaluates to v at rho
    assert len(b["P"]) == 1 << len(rho) and sc.mle_eval(b["P"], rho, p) == v
    # every reduced claim is the claimed polynomial's own evaluation
    s_max = max(shape(I)[0] for I in insts)
    for I, (s, _, _), c in zip(insts, [shape(I) for I in insts], proof["claims"]):
        assert c[3] == sc.mle_eval(I["E"] + [0] * ((1 << s) - I["rows"]), proof["rx"][s_max - s:], p)


def test_batched_verifiers_reject_tampering(spec, instances):
    p = spec.FIELD_MODULUS[0]
    insts = instances[:2]
    good = python_batched_prover(insts, challenge, p)
    assert check(insts, good, p) is not None
    # one flipped bit of one instance's E: that instance no longer satisfies the relaxed R1CS
    bad = [insts[0], dict(insts[1], E=[insts[1]["E"][0] ^ 1] + insts[1]["E"][1:])]
    assert check(insts, python_batched_prover(bad, challenge, p), p) is None
    # the transcript replayed against a changed u of one instance
    assert check([insts[0], dict(insts[1], u=(insts[1]["u"] + 1) % p)], good, p) is None
    # two instances swapped
    assert check(insts[::-1], good, p) is None
    assert check(insts[::-1], python_batched_prover(insts[::-1], challenge, p), p) is not None
    # a wrong reduced evaluation left_j
    for j in (0, 3):
        left = list(good["batch"]["left"])
        left[j] = (left[j] + 1) % p
        assert check(insts, dict(good, batch=dict(good["batch"], left=left)), p) is None


def test_poly_combine_rejects_bad_arguments_and_has_no_cpu_fallback(L):
    """argument checks of lurk_poly_combine_dev run before any device work; valid arguments without a GPU give LURK_ERR_NOGPU"""
    import ctypes as C
    lib, E = L._capi.lib(), L._capi
    a, b, out = (np.zeros(32 * 16, dtype=np.uint8) for _ in range(3))
    ptrs = (C.c_void_p * 2)(C.c_void_p(a.ctypes.data), C.c_void_p(b.ctypes.data))
    lens = (C.c_size_t * 2)(16, 4)
    co = np.zeros(64, dtype=np.uint8)
    co[0] = co[32] = 1
    dout = C.c_void_p(out.ctypes.data)
    call = lambda n=2, ptrs=ptrs, lens=lens, co=co, dout=dout, out_len=16, field=0: lib.lurk_poly_combine_dev(
        field, n, ptrs, lens, E.np_ptr(co) if co is not None else None, dout, out_len, E.FMT_CANONICAL, None)
    assert call(n=0) == E.ERR_ARG
    assert call(n=121) == E.ERR_ARG
    assert call(out_len=8) == E.ERR_ARG                                                           # len_0 > out_len
    assert call(ptrs=(C.c_void_p * 2)(C.c_void_p(a.ctypes.data), None)) == E.ERR_ARG
    assert call(ptrs=None) == E.ERR_ARG and call(lens=None) == E.ERR_ARG and call(co=None) == E.ERR_ARG and call(dout=None) == E.ERR_ARG
    assert call(dout=C.c_void_p(a.ctypes.data + 32 * 15)) == E.ERR_ARG                            # output overlaps an input
    assert call(field=9) == E.ERR_ARG
    unreduced = co.copy()
    unreduced[32:64] = 0xff
    assert call(co=unreduced) == E.ERR_RANGE
    assert len(lib.lurk_last_error()) > 0
    if lib.lurk_device_count() == 0:
        assert call() == E.ERR_NOGPU
