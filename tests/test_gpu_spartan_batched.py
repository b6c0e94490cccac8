"""SuperNova's `compress` on the GPU (lurk-beta_b200/spartan.py: BatchedRelaxedR1CSProver + batch_eval_prove, csrc/combine.cu:
lurk_poly_combine_dev): the running instances of all NIVC circuits proven in one batched Spartan argument, every evaluation claim
reduced to one claim about one joint polynomial, and that polynomial opened ONCE -- HyperKZG on BN254 under a powers-of-tau key of
known beta (oracle/kzg.py: verify_known_beta), IPA on Grumpkin.  Checked by the verifiers of tests/spartan_batched_oracle.py,
end to end from a GPU fold of two NIVC circuits.  Reference: src/proof/supernova.rs:110,293-317, nova.rs:92."""
import hashlib

import numpy as np
import pytest

from oracle import kzg, nifs, spartan as ospartan, sumcheck as sc
from spartan_batched_oracle import batch_eval_verify, eval_claims, python_batched_prover, shape, verify_batched
from test_gpu_fold_pipeline import _build, _fill, _layout, _step_inputs
from test_gpu_spartan_chain import challenge, rows_of, to_device
from test_oracle_spartan_batched import SHAPES, instance
from util import ints, pack, random_elements

pytestmark = pytest.mark.gpu
CURVE, FIELD = 0, 0
BETA = 0x1234567890abcdef1234567890abcdef


def to_canonical_ints(L, field, t):
    import ctypes as C
    c = t.clone()
    L._capi.check(L._capi.lib().lurk_convert_dev(field, C.c_void_p(c.data_ptr()), c.numel() // 32, L.FMT_CANONICAL, C.c_void_p(c.data_ptr()), None))
    return ints(c.cpu().numpy())


def kzg_key(L, spec, n):
    pb = spec.FIELD_MODULUS[spec.CURVES[CURVE]["base"]]
    g = spec.ec_mul(4242, spec.CURVES[CURVE]["gen"], pb)
    return g, L.CommitmentKey.powers_of_tau(CURVE, g, BETA % spec.FIELD_MODULUS[FIELD], n)


def hyperkzg_open(L, ck):
    """the `open` callback of batch_eval_prove: HyperKZG on the joint polynomial, keeping the PCS transcript for the check"""
    p = int.from_bytes(L.spartan.field_modulus(FIELD), "little")

    def open_(d_P, point, value):
        log = []

        def cb(rnd, msg):
            log.append(bytes(msg))
            return challenge("pcs", (rnd, bytes(msg))) % p
        com, v, w = L.spartan.hyperkzg_prove(CURVE, ck, d_P.data_ptr(), point, cb)
        return dict(com=com, v=v, w=w, log=log)
    return open_


def kzg_accepts(spec, g, polys, gp, c0, rho, v, op):
    """the verifier's algebra of the one opening, commitments as discrete logs (key beta^i g).  c0: the scalar of the joint commitment
    sum_j gamma^j comm_j, derived by the caller from the per-claim commitments.  Also checks that the prover's commitments are those
    of the joint polynomial sum_j gamma^j P_j (zero-extended)."""
    p, pb = spec.FIELD_MODULUS[FIELD], spec.FIELD_MODULUS[spec.CURVES[CURVE]["base"]]
    beta = BETA % p
    joint = [0] * (1 << len(rho))
    for c, P in zip(gp, polys):
        for i, x in enumerate(P):
            joint[i] = (joint[i] + c * x) % p
    at_beta = [kzg.poly_eval(f, beta, p) for f in kzg.fold_chain(joint, rho, p)]
    assert op["com"] == [spec.ec_mul(s, g, pb) for s in at_beta[1:]]
    r, q = challenge("pcs", (0, op["log"][0])) % p, challenge("pcs", (1, op["log"][1])) % p
    u = [r, (-r) % p, r * r % p]
    Bbeta = sum(pow(q, j, p) * s for j, s in enumerate([c0] + at_beta[1:])) % p
    w_scalars = [(Bbeta - sum(pow(q, j, p) * op["v"][t][j] for j in range(len(rho)))) * pow(beta - u[t], -1, p) % p for t in range(3)]
    if op["w"] != [spec.ec_mul(s, g, pb) for s in w_scalars]:
        return False
    return kzg.verify_known_beta(CURVE, g, beta, c0, rho, v, at_beta[1:], op["v"], w_scalars, r, q)


def reduced(insts, proof, p):
    ok, rx, ry = verify_batched(insts, proof, challenge, p)
    if not ok:
        return None
    pts = eval_claims(insts, proof, rx, ry)
    b = proof["batch"]
    return batch_eval_verify(b["rounds"], [x for x, _ in pts], [v for _, v in pts], b["left"], challenge, p)


def padded_polys(insts):
    """the 2k polynomials of the reduction, in its order: W_i padded to num_vars_i, then E_i padded to 2^s_i"""
    sh = [shape(I) for I in insts]
    return ([I["W"] + [0] * (nv - I["n_w"]) for I, (_, nv, _) in zip(insts, sh)]
            + [I["E"] + [0] * ((1 << s) - I["rows"]) for I, (s, _, _) in zip(insts, sh)])


def test_poly_combine_matches_oracle(L, spec):
    import torch
    p = spec.FIELD_MODULUS[FIELD]
    lens = [1, 1 << 5, 1 << 12, 1 << 17]
    bufs = [random_elements(FIELD, n, seed=10 + j) for j, n in enumerate(lens)]
    coeffs = ints(random_elements(FIELD, len(lens), seed=9))
    dev = [to_device(L, FIELD, b) for b in bufs]
    for out_len in (1 << 17, (1 << 17) + 3001):
        out = torch.full((out_len * 32,), 0xAB, dtype=torch.uint8, device="cuda")
        L.spartan.poly_combine(FIELD, [(d.data_ptr(), n) for d, n in zip(dev, lens)], coeffs, out.data_ptr(), out_len)
        want = [0] * out_len
        for c, b in zip(coeffs, bufs):
            for i, x in enumerate(ints(b)):
                want[i] = (want[i] + c * x) % p
        assert to_canonical_ints(L, FIELD, out) == want
    # the inputs are read, not modified
    assert all(np.array_equal(to_canonical_ints(L, FIELD, d), ints(b)) for d, b in zip(dev, bufs))


@pytest.fixture(scope="module")
def instances(oracle, spec):
    return [instance(oracle, spec, 31 + i, shp) for i, shp in enumerate(SHAPES)]


def gpu_inputs(L, insts):
    provers, inputs = [], []
    for I in insts:
        pr = L.spartan.RelaxedR1CSProver(FIELD, I["mats"], I["n_w"], len(I["X"]))
        z = pr.pad_z(to_device(L, FIELD, pack(I["W"])), I["u"], I["X"])
        provers.append(pr)
        inputs.append((z, to_device(L, FIELD, pack(I["E"])), I["u"], I["X"]))
    return L.spartan.BatchedRelaxedR1CSProver(provers), inputs


def test_batched_chain_is_accepted_and_opens_once(L, oracle, spec, instances):
    p = spec.FIELD_MODULUS[FIELD]
    insts = list(instances)
    prover, inputs = gpu_inputs(L, insts)
    m_max = max(max(s, t - 1) for s, _, t in (shape(I) for I in insts))
    g, ck = kzg_key(L, spec, 1 << m_max)
    timings = {}
    proof = prover.prove(inputs, challenge, hyperkzg_open(L, ck), timings)
    # the GPU transcript is the pure-Python prover's, challenge for challenge
    want = python_batched_prover(insts, challenge, p)
    for key in ("outer_rounds", "inner_rounds", "claims", "eval_W", "rx", "ry"):
        assert [tuple(x) if isinstance(x, (list, tuple)) else x for x in proof[key]] == \
               [tuple(x) if isinstance(x, (list, tuple)) else x for x in want[key]], key
    for key in ("rounds", "rho", "left", "gamma", "v"):
        assert proof["batch"][key] == want["batch"][key], key
    got = reduced(insts, proof, p)
    assert got is not None
    rho, v, gp = got
    polys = padded_polys(insts)
    c0 = sum(c * kzg.poly_eval(P, BETA % p, p) for c, P in zip(gp, polys)) % p
    op = proof["batch"]["opening"]
    assert kzg_accepts(spec, g, polys, gp, c0, rho, v, op)
    assert not kzg_accepts(spec, g, polys, gp, c0, rho, (v + 1) % p, op)
    assert not kzg_accepts(spec, g, polys, gp, (c0 + 1) % p, rho, v, op)
    assert set(timings) >= {"outer sum-check", "inner sum-check", "batch_eval_reduce + opening"}
    # tampering: a flipped bit of one instance's E, a changed u, swapped instances, a wrong reduced evaluation
    bad_E = pack(insts[1]["E"])
    bad_E[0] ^= 1
    bad_inputs = list(inputs)
    bad_inputs[1] = (inputs[1][0], to_device(L, FIELD, bad_E), inputs[1][2], inputs[1][3])
    assert reduced(insts, prover.prove(bad_inputs, challenge, hyperkzg_open(L, ck)), p) is None
    assert reduced([insts[0], dict(insts[1], u=(insts[1]["u"] + 1) % p), insts[2]], proof, p) is None
    assert reduced([insts[1], insts[0], insts[2]], proof, p) is None
    left = list(proof["batch"]["left"])
    left[4] = (left[4] + 1) % p
    assert reduced(insts, dict(proof, batch=dict(proof["batch"], left=left)), p) is None


def test_nova_single_instance_opens_once(L, oracle, spec, instances):
    """the Nova chain (k = 1): RelaxedR1CSProver.prove, unchanged, then batch_eval_prove over (W, ry[1:]) and (E, rx): one opening"""
    p = spec.FIELD_MODULUS[FIELD]
    I = instances[0]
    pr = L.spartan.RelaxedR1CSProver(FIELD, I["mats"], I["n_w"], 2)
    z = pr.pad_z(to_device(L, FIELD, pack(I["W"])), I["u"], I["X"])
    proof = pr.prove(z, to_device(L, FIELD, pack(I["E"])), I["u"], challenge)
    ok, rx, ry = ospartan.verify(I["R"], I["n_w"], pr.num_vars, pr.log_rows, I["u"], I["X"], proof, challenge, p)
    assert ok
    g, ck = kzg_key(L, spec, max(pr.num_vars, 1 << pr.log_rows))
    b = L.spartan.batch_eval_prove(FIELD, [(z, ry[1:], proof["eval_W"]), (proof["E_padded"], rx, proof["claims"][3])], challenge, hyperkzg_open(L, ck))
    got = batch_eval_verify(b["rounds"], [ry[1:], rx], [proof["eval_W"], proof["claims"][3]], b["left"], challenge, p)
    assert got is not None
    rho, v, gp = got
    assert (rho, v) == (b["rho"], b["v"])
    polys = padded_polys([I])
    c0 = sum(c * kzg.poly_eval(P, BETA % p, p) for c, P in zip(gp, polys)) % p
    assert kzg_accepts(spec, g, polys, gp, c0, rho, v, b["opening"])
    assert not kzg_accepts(spec, g, polys, gp, c0, rho, (v + 1) % p, b["opening"])


def test_fold_then_compress_from_device_resident_running_instances(L, oracle, spec):
    """two NIVC circuits folded on the GPU under the powers-of-tau key, compressed straight from LURK_FOLD_BUF_Z1 / E1; the verifier's
    joint commitment is built from the fold context's own comm_W / comm_E"""
    p, pb = spec.FIELD_MODULUS[FIELD], spec.FIELD_MODULUS[spec.CURVES[CURVE]["base"]]
    rng = np.random.default_rng(5)
    shapes = ((30, 25), (38, 7))                                      # (glue, linear rows) of the two circuits, one frame each
    slot_elems = _layout(oracle, 1, 0)["slot_elems"]
    n_key = max(1 << max(1, (max(slot_elems + glue, 3) - 1).bit_length()) for glue, _ in shapes)     # the longest W (num_vars) ...
    n_key = max([n_key] + [1 << max(1, (2 * glue + lin - 1).bit_length()) for glue, lin in shapes])  # ... or padded E
    g, ck = kzg_key(L, spec, n_key)
    ctxs, lays, matss, glues, bis = [], [], [], [], []
    for glue, lin in shapes:
        ctx, lay, mats, n_w, rows, glue_fn, _, _, bi = _build(L, oracle, nifs, spec, rng, frames=1, glue=glue, lin_rows=lin, bases="pot", ck=ck)
        assert max(n_w, rows) <= n_key
        ctxs.append(ctx), lays.append(lay), matss.append(mats), glues.append(glue_fn), bis.append(bi)
    nivc = L.SuperNovaFoldContext(ctxs)
    for s, ci in enumerate([0, 1, 0, 1, 1, 0]):
        b = nivc._next[ci]
        _fill(ctxs[ci], b, lays[ci], _step_inputs(oracle, nifs, spec, lays[ci], glues[ci], 40 + s, rng), 5, bis[ci])
        assert nivc.stage_a(ci) == b
        nivc.fold(ci, b)
        nivc.collect(ci, b)
    runs = [c.get_running() for c in ctxs]
    assert all(c.check_running() == (0, True, True) for c in ctxs)
    provers = [L.spartan.RelaxedR1CSProver(FIELD, mats, c.n_w, 2) for mats, c in zip(matss, ctxs)]
    inputs = [L.spartan.fold_running_inputs(pr, c) for pr, c in zip(provers, ctxs)]
    for (_, _, u, X), run in zip(inputs, runs):
        assert [u] == nifs.ints(run["u"]) and X == nifs.ints(run["X"]) and u != 1
    proof = L.spartan.BatchedRelaxedR1CSProver(provers).prove(inputs, challenge, hyperkzg_open(L, ck))
    # verifier side: the public instances (matrices, u, X, commitments) only
    insts = [dict(R=[rows_of(m) for m in mats], n_w=c.n_w, rows=c.n_rows, u=nifs.ints(run["u"])[0], X=nifs.ints(run["X"])) for mats, c, run in zip(matss, ctxs, runs)]
    got = reduced(insts, proof, p)
    assert got is not None
    rho, v, gp = got
    comms = [nifs.point_of(run["comm_W"]) for run in runs] + [nifs.point_of(run["comm_E"]) for run in runs]
    joint_comm = None
    for c, P in zip(gp, comms):
        joint_comm = spec.ec_add(joint_comm, spec.ec_mul(c, P, pb), pb)
    # the discrete log of the joint commitment (key of known beta), from the running witness the fold kept
    polys = padded_polys([dict(I, W=nifs.ints(run["W"]), E=nifs.ints(run["E"])) for I, run in zip(insts, runs)])
    c0 = sum(c * kzg.poly_eval(P, BETA % p, p) for c, P in zip(gp, polys)) % p
    assert joint_comm == spec.ec_mul(c0, g, pb)
    assert kzg_accepts(spec, g, polys, gp, c0, rho, v, proof["batch"]["opening"])
    assert not kzg_accepts(spec, g, polys, gp, c0, rho, (v + 1) % p, proof["batch"]["opening"])


def test_secondary_reduction_ends_in_one_ipa_opening(L, oracle, spec):
    """field 1 / Grumpkin: the k = 1 reduction of (W at a 5-point, E at a 6-point) opened by ipa_prove with b = eq(rho); the IPA relation
    commit(a'; G') + a' b' ck_c = P + sum_i (r_i^2 L_i + r_i^-2 R_i), P = sum_j gamma^j comm_j + v ck_c, holds"""
    import torch
    curve = 1
    Cv = spec.CURVES[curve]
    field = Cv["scalar"]
    pb, q = spec.FIELD_MODULUS[Cv["base"]], spec.FIELD_MODULUS[field]
    ms = [5, 6]
    bufs = [random_elements(field, 1 << m, seed=20 + m) for m in ms]
    polys = [ints(b) for b in bufs]
    points = [ints(random_elements(field, m, seed=30 + m)) for m in ms]
    values = [sc.mle_eval(P, x, q) for P, x in zip(polys, points)]
    n = 1 << max(ms)
    bases = oracle.gen_bases(curve, n + 1, start=5)
    Gs = list(zip(ints(bases)[0::2], ints(bases)[1::2]))
    G, gc = Gs[:n], Gs[n]
    ck = L.CommitmentKey(curve, bases[:64 * n])

    def chal(rnd, msg):
        return 1 + int.from_bytes(hashlib.sha256(bytes([rnd]) + msg).digest()[:16], "little")

    def open_(d_P, rho, v):
        eq = torch.empty_like(d_P)
        L.spartan.eq_evals(field, rho, eq.data_ptr())
        return L.spartan.ipa_prove(curve, ck, gc, d_P.data_ptr(), eq.data_ptr(), len(rho), chal)

    dev = [to_device(L, field, b) for b in bufs]
    b = L.spartan.batch_eval_prove(field, [(d, x, v) for d, x, v in zip(dev, points, values)], challenge, open_)
    got = batch_eval_verify(b["rounds"], points, values, b["left"], challenge, q)
    assert got is not None
    rho, v, gp = got
    add = lambda P, Q: spec.ec_add(P, Q, pb)
    mul = lambda k, P: spec.ec_mul(k % q, P, pb)
    acc = mul(v, gc)
    for c, P in zip(gp, polys):
        acc = add(acc, mul(c, spec.msm_naive(curve, G[:len(P)], P)))
    Ls, Rs, a_fin, b_fin = b["opening"]
    bvec = sc.eq_evals(rho, q)
    enc = lambda P: (pack([P[0], P[1], 1]) if P is not None else np.zeros(96, dtype=np.uint8)).tobytes()
    for rnd in range(len(rho)):
        r = chal(rnd, enc(Ls[rnd]) + enc(Rs[rnd]))
        ri = pow(r, -1, q)
        acc = add(acc, add(mul(r * r, Ls[rnd]), mul(ri * ri, Rs[rnd])))
        bvec = sc.ipa_fold_scalars(bvec, ri, r, q)
        G = sc.ipa_fold_bases(curve, G, ri, r)
    assert b_fin == bvec[0]
    assert add(mul(a_fin, G[0]), mul(a_fin * b_fin, gc)) == acc
    # the inputs of the reduction are not consumed
    assert all(to_canonical_ints(L, field, d) == P for d, P in zip(dev, polys))
