"""The verifier's side of SuperNova's `compress` (Arecibo spartan::batched::BatchedRelaxedR1CSSNARK, reference
src/proof/supernova.rs:110,293-317) and of batch_eval_reduce (spartan/mod.rs), restated from the public crate with the transcript
replaced by an explicit challenge function, plus a pure-Python prover that follows the same list as the GPU prover
(lurk-beta_b200/spartan.py: BatchedRelaxedR1CSProver, batch_eval_prove).  Built on oracle/spartan.py and oracle/sumcheck.py.

Instance i has rows padded to 2^s_i and z of 2^t_i = 2 num_vars_i elements; it joins each batched sum-check late and uses the
suffix of the shared challenge vector (r_x_i = r_x[s_max - s_i:], r_y_i = r_y[t_max - t_i:]).  The first claim of a batched
sum-check is sum_i c_i 2^(max - n_i) claim_i, as in oracle/sumcheck.py: prove_batch.

Parity: UNPINNED against Arecibo's proof bytes; pinned by construction (the verifiers accept the provers' output, a perturbed
instance or evaluation is rejected)."""
from oracle import spartan as osp, sumcheck as sc


def powers(x, n, p):
    out = [1]
    for _ in range(n - 1):
        out.append(out[-1] * x % p)
    return out[:n]


def eq_at(x, y, p):
    acc = 1
    for a, b in zip(x, y):
        acc = acc * (a * b + (1 - a) * (1 - b)) % p
    return acc


def shape(inst):
    """(s, num_vars, t) as RelaxedR1CSProver derives them"""
    s = max(1, (inst["rows"] - 1).bit_length())
    nv = 1 << max(1, (max(inst["n_w"], len(inst["X"]) + 1) - 1).bit_length())
    return s, nv, nv.bit_length()


def _io(inst, p):
    return (inst["u"] % p, [x % p for x in inst["X"]])


# ------------------------------------------------------------------------------------------------ provers
def batch_eval_prove(polys, points, values, challenge, p):
    """batch_eval_reduce over claims P_j(points_j) = values_j (polys: full 2^len(point) evaluation lists)"""
    n = len(polys)
    ms = [len(x) for x in points]
    m = max(ms)
    sigma = challenge("batch_r", [v % p for v in values]) % p
    rounds, rho, fin, _ = sc.prove_batch([[list(P), sc.eq_evals(x, p)] for P, x in zip(polys, points)], "quad", values, powers(sigma, n, p),
                                         lambda i, ev: challenge("batch", (i, ev)), p)
    left = [f[0] for f in fin]
    gamma = challenge("batch_g", left) % p
    gp = powers(gamma, n, p)
    joint = [0] * (1 << m)
    v = 0
    for g, P, mj, lj in zip(gp, polys, ms, left):
        for i, c in enumerate(P):
            joint[i] = (joint[i] + g * c) % p
        v = (v + g * eq_at([0] * (m - mj), rho[:m - mj], p) * lj) % p
    return dict(rounds=rounds, rho=rho, values=[v % p for v in values], left=left, gamma=gamma, v=v, P=joint)


def python_batched_prover(insts, challenge, p):
    """insts: dicts R (rows of A, B, C: oracle/spartan.py matrices_eval form), n_w, rows, W, E, u, X (ints).  Returns the transcript the
    GPU prover returns, with the reduction under "batch"."""
    k = len(insts)
    sh = [shape(I) for I in insts]
    s_max, t_max = max(s for s, _, _ in sh), max(t for _, _, t in sh)
    zs, prods, Eps = [], [], []
    for I, (s, nv, _) in zip(insts, sh):
        z = I["W"] + [0] * (nv - I["n_w"]) + [I["u"]] + I["X"] + [0] * (nv - 1 - len(I["X"]))

        def mv(rowsl):
            return [sum(v * z[osp.col_map(c, I["n_w"], nv)] for c, v in r) % p for r in rowsl] + [0] * ((1 << s) - I["rows"])
        Az, Bz, Cz = [mv(r) for r in I["R"]]
        Ep = I["E"] + [0] * ((1 << s) - I["rows"])
        zs.append(z)
        prods.append((Az, Bz, Cz, [(I["u"] * c + e) % p for c, e in zip(Cz, Ep)]))
        Eps.append(Ep)
    rho = challenge("outer_r", [_io(I, p) for I in insts]) % p
    tau = [challenge("tau", t) % p for t in range(s_max)]
    outer = sc.prove_batch([[sc.eq_evals(tau[s_max - s:], p), Az, Bz, uCzE] for (s, _, _), (Az, Bz, _, uCzE) in zip(sh, prods)], "cubic", [0] * k,
                           powers(rho, k, p), lambda i, ev: challenge("outer", (i, ev)), p)
    rx = outer[1]
    claims = []
    for i, ((s, _, _), (_, _, Cz, _), Ep) in enumerate(zip(sh, prods, Eps)):
        eqrx = sc.eq_evals(rx[s_max - s:], p)
        claims.append((outer[2][i][1], outer[2][i][2], sc.inner_product(Cz, eqrx, p), sc.inner_product(Ep, eqrx, p)))
    r = challenge("inner_r", claims) % p
    abcs = []
    for I, (s, nv, _) in zip(insts, sh):
        eqrx = sc.eq_evals(rx[s_max - s:], p)
        abc = [0] * (2 * nv)
        for m, rowsl in enumerate(I["R"]):
            for i, row in enumerate(rowsl):
                for c, v in row:
                    j = osp.col_map(c, I["n_w"], nv)
                    abc[j] = (abc[j] + pow(r, m, p) * eqrx[i] * v) % p
        abcs.append(abc)
    joints = [(c[0] + r * c[1] + r * r * c[2]) % p for c in claims]
    inner = sc.prove_batch([[abc, z] for abc, z in zip(abcs, zs)], "quad", joints, powers(r * r * r % p, k, p),
                           lambda i, ev: challenge("inner", (i, ev)), p)
    ry = inner[1]
    Wps = [I["W"] + [0] * (nv - I["n_w"]) for I, (_, nv, _) in zip(insts, sh)]
    eval_W = [sc.mle_eval(Wp, ry[t_max - t + 1:], p) for Wp, (_, _, t) in zip(Wps, sh)]
    batch = batch_eval_prove(Wps + Eps, [ry[t_max - t + 1:] for _, _, t in sh] + [rx[s_max - s:] for s, _, _ in sh],
                             eval_W + [c[3] for c in claims], challenge, p)
    return dict(outer_rounds=outer[0], inner_rounds=inner[0], claims=claims, eval_W=eval_W, rx=rx, ry=ry, batch=batch)


# ------------------------------------------------------------------------------------------------ verifiers
def verify_batched(insts, proof, challenge, p):
    """insts: dicts R, n_w, rows, u, X.  Checks the outer sum-check against sum_i rho^i eq(tau_i, r_x_i) (Az Bz - u Cz - E)_i and the
    inner one against sum_i (r^3)^i (eA + r eB + r^2 eC)_i z_i(r_y_i), the matrix MLEs evaluated from the matrices.
    Returns (ok, rx, ry); eval_W_i at r_y_i[1:] and E_i(r_x_i) remain to be checked against the commitments (eval_claims)."""
    k = len(insts)
    sh = [shape(I) for I in insts]
    s_max, t_max = max(s for s, _, _ in sh), max(t for _, _, t in sh)
    if len(proof["claims"]) != k or len(proof["eval_W"]) != k:
        return False, None, None
    rho = challenge("outer_r", [_io(I, p) for I in insts]) % p
    tau = [challenge("tau", t) % p for t in range(s_max)]
    rx = [challenge("outer", (i, ev)) % p for i, ev in enumerate(proof["outer_rounds"])]
    last = sc.verify(proof["outer_rounds"], rx, 0, 3, p)
    if last is None or len(rx) != s_max:
        return False, None, None
    want = 0
    for c, I, (s, _, _), (cA, cB, cC, cE) in zip(powers(rho, k, p), insts, sh, proof["claims"]):
        want += c * eq_at(tau[s_max - s:], rx[s_max - s:], p) * (cA * cB - I["u"] * cC - cE)
    if last != want % p:
        return False, None, None
    r = challenge("inner_r", proof["claims"]) % p
    co = powers(r * r * r % p, k, p)
    claim = sum(c * (1 << (t_max - t)) * (cA + r * cB + r * r * cC) for c, (_, _, t), (cA, cB, cC, _) in zip(co, sh, proof["claims"])) % p
    ry = [challenge("inner", (i, ev)) % p for i, ev in enumerate(proof["inner_rounds"])]
    last2 = sc.verify(proof["inner_rounds"], ry, claim, 2, p)
    if last2 is None or len(ry) != t_max:
        return False, None, None
    want2 = 0
    for c, I, (s, nv, t), ew in zip(co, insts, sh, proof["eval_W"]):
        ryi = ry[t_max - t:]
        eA, eB, eC = osp.matrices_eval(I["R"], I["n_w"], nv, rx[s_max - s:], ryi, p)
        tail = [I["u"] % p] + [x % p for x in I["X"]]
        eval_X = sc.mle_eval(tail + [0] * (nv - len(tail)), ryi[1:], p)
        want2 += c * (eA + r * eB + r * r * eC) * ((1 - ryi[0]) * ew + ryi[0] * eval_X)
    if last2 != want2 % p:
        return False, None, None
    return True, rx, ry


def eval_claims(insts, proof, rx, ry):
    """the 2k (point, value) claims the reduction takes, in its order: W_i at r_y_i[1:], then E_i at r_x_i"""
    sh = [shape(I) for I in insts]
    s_max, t_max = max(s for s, _, _ in sh), max(t for _, _, t in sh)
    return ([(ry[t_max - t + 1:], ew) for (_, _, t), ew in zip(sh, proof["eval_W"])]
            + [(rx[s_max - s:], c[3]) for (s, _, _), c in zip(sh, proof["claims"])])


def batch_eval_verify(rounds, points, values, left, challenge, p):
    """batch_eval_reduce's verifier: the sum-check of sum_j sigma^j P_j(x) eq(points_j, x) ends in sum_j sigma^j eq(points_j, rho_j) left_j
    (rho_j the suffix of rho of point j's length).  Returns (rho, v, gamma powers) -- the joint polynomial sum_j gamma^j P_j must open
    to v at rho under the joint commitment sum_j gamma^j comm_j -- or None."""
    n = len(points)
    if len(values) != n or len(left) != n:
        return None
    ms = [len(x) for x in points]
    m = max(ms)
    values = [v % p for v in values]
    sp = powers(challenge("batch_r", values) % p, n, p)
    claim = sum(c * (1 << (m - mj)) * v for c, mj, v in zip(sp, ms, values)) % p
    rho = [challenge("batch", (i, ev)) % p for i, ev in enumerate(rounds)]
    last = sc.verify(rounds, rho, claim, 2, p)
    if last is None or len(rho) != m:
        return None
    if last != sum(c * eq_at(x, rho[m - mj:], p) * lj for c, x, mj, lj in zip(sp, points, ms, left)) % p:
        return None
    gp = powers(challenge("batch_g", list(left)) % p, n, p)
    v = sum(g * eq_at([0] * (m - mj), rho[:m - mj], p) * lj for g, mj, lj in zip(gp, ms, left)) % p
    return rho, v, gp
