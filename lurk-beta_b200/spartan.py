"""Host-side mirror of the Arecibo interfaces behind `compress` (reference src/proof/nova.rs:341-356 -> CompressedSNARK::prove
-> spartan::snark::RelaxedR1CSSNARK::prove): SumcheckProof::prove_quad / prove_cubic_with_additive_term, EqPolynomial::evals,
MultilinearPolynomial::evaluate and provider::ipa_pc::InnerProductArgument::prove, all on device-resident vectors through the C ABI
(include/lurk_b200.h, N4).  The transcript is the caller's: `challenge(round, message_bytes) -> int`."""
import ctypes as C

import numpy as np

from . import _capi

QUAD, CUBIC = _capi.SUMCHECK_QUAD, _capi.SUMCHECK_CUBIC


def _callback(challenge, errors):
    def cb(user, rnd, msg, msg_len, out):
        try:
            r = int(challenge(rnd, bytes(msg[i] for i in range(msg_len))))
            for i, byte in enumerate(r.to_bytes(32, "little")):
                out[i] = byte
            return 0
        except Exception as e:          # never unwind through the C frames
            errors.append(e)
            return 1
    return _capi.CHALLENGE_FN(cb)


def _ints(buf):
    return [int.from_bytes(buf[i:i + 32].tobytes(), "little") for i in range(0, buf.size, 32)]


def _fe(x):
    return np.frombuffer(int(x).to_bytes(32, "little"), dtype=np.uint8).copy()


def sumcheck_prove(field_id, kind, poly_ptrs, num_rounds, claim, challenge, stream=0):
    """poly_ptrs: device pointers of the 2 (QUAD) or 4 (CUBIC) polynomials, 2^num_rounds Montgomery elements each (consumed).
    claim: int.  challenge(round, message) -> int (canonical).  Returns (round_evals [[int]], challenges [int], final_evals [int])."""
    k, deg1 = (2, 3) if kind == QUAD else (4, 4)
    ptrs = (C.c_void_p * k)(*[C.c_void_p(p) for p in poly_ptrs])
    rounds = np.zeros(max(1, num_rounds) * deg1 * 32, dtype=np.uint8)
    chal = np.zeros(max(1, num_rounds) * 32, dtype=np.uint8)
    fin = np.zeros(k * 32, dtype=np.uint8)
    errors = []
    cb = _callback(challenge, errors)
    rc = _capi.lib().lurk_sumcheck_prove_dev(field_id, kind, ptrs, num_rounds, _capi.np_ptr(_fe(claim)), cb, None, _capi.np_ptr(rounds),
                                             _capi.np_ptr(chal), _capi.np_ptr(fin), _capi.FMT_CANONICAL, C.c_void_p(stream))
    if errors:
        raise errors[0]
    _capi.check(rc)
    ev = _ints(rounds)
    return [ev[i * deg1:(i + 1) * deg1] for i in range(num_rounds)], _ints(chal)[:num_rounds], _ints(fin)


def sumcheck_prove_batch(field_id, kind, instances, claims, coeffs, challenge, stream=0):
    """SumcheckProof::prove_*_batch.  instances: [(poly_ptrs, num_rounds)], claims / coeffs: ints.
    Returns (round_evals, challenges, final_evals per instance)."""
    k, deg1 = (2, 3) if kind == QUAD else (4, 4)
    n = len(instances)
    flat = [p for ptrs, _ in instances for p in ptrs]
    ptrs = (C.c_void_p * (n * k))(*[C.c_void_p(p) for p in flat])
    nr = (C.c_int * n)(*[r for _, r in instances])
    mx = max(r for _, r in instances)
    rounds = np.zeros(max(1, mx) * deg1 * 32, dtype=np.uint8)
    chal = np.zeros(max(1, mx) * 32, dtype=np.uint8)
    fin = np.zeros(n * k * 32, dtype=np.uint8)
    cl = np.concatenate([_fe(c) for c in claims])
    co = np.concatenate([_fe(c) for c in coeffs])
    errors = []
    cb = _callback(challenge, errors)
    rc = _capi.lib().lurk_sumcheck_prove_batch_dev(field_id, kind, n, ptrs, nr, _capi.np_ptr(cl), _capi.np_ptr(co), cb, None, _capi.np_ptr(rounds),
                                                   _capi.np_ptr(chal), _capi.np_ptr(fin), _capi.FMT_CANONICAL, C.c_void_p(stream))
    if errors:
        raise errors[0]
    _capi.check(rc)
    ev, fi = _ints(rounds), _ints(fin)
    return [ev[i * deg1:(i + 1) * deg1] for i in range(mx)], _ints(chal)[:mx], [fi[i * k:(i + 1) * k] for i in range(n)]


def eq_evals(field_id, tau, d_out_ptr, out_fmt=_capi.FMT_MONTGOMERY, stream=0):
    """EqPolynomial::new(tau).evals() into device memory (2^len(tau) elements in out_fmt); tau: ints"""
    R = 1 << 256
    if out_fmt == _capi.FMT_MONTGOMERY:
        p = int.from_bytes(field_modulus(field_id), "little")
        tau = [t * R % p for t in tau]
    buf = np.frombuffer(b"".join(int(t).to_bytes(32, "little") for t in tau) or bytes(32), dtype=np.uint8).copy()
    _capi.check(_capi.lib().lurk_eq_evals_dev(field_id, _capi.np_ptr(buf), len(tau), C.c_void_p(d_out_ptr), out_fmt, C.c_void_p(stream)))


def field_modulus(field_id):
    out = np.zeros(32, dtype=np.uint8)
    _capi.check(_capi.lib().lurk_field_modulus(field_id, _capi.np_ptr(out)))
    return out.tobytes()


def inner_product(field_id, d_a_ptr, d_b_ptr, n, stream=0):
    out = np.zeros(32, dtype=np.uint8)
    _capi.check(_capi.lib().lurk_inner_product_dev(field_id, C.c_void_p(d_a_ptr), C.c_void_p(d_b_ptr), n, _capi.np_ptr(out),
                                                   _capi.FMT_CANONICAL, C.c_void_p(stream)))
    return int.from_bytes(out.tobytes(), "little")


def poly_combine(field_id, polys, coeffs, d_out_ptr, out_len, stream=0):
    """PolyEvalWitness::batch_diff_size: out[i] = sum_j coeffs[j] P_j[i], every P_j zero-extended at the end to out_len elements.
    polys: [(device pointer, length)] of Montgomery elements; coeffs: ints; d_out_ptr: out_len elements, not overlapping any P_j."""
    n = len(polys)
    ptrs = (C.c_void_p * n)(*[C.c_void_p(ptr) for ptr, _ in polys])
    lens = (C.c_size_t * n)(*[int(ln) for _, ln in polys])
    co = np.concatenate([_fe(c) for c in coeffs]) if coeffs else np.zeros(32, dtype=np.uint8)
    _capi.check(_capi.lib().lurk_poly_combine_dev(field_id, n, ptrs, lens, _capi.np_ptr(co), C.c_void_p(d_out_ptr), out_len, _capi.FMT_CANONICAL,
                                                  C.c_void_p(stream)))


def ipa_fold_scalars(field_id, d_a_ptr, n, x, y, stream=0):
    _capi.check(_capi.lib().lurk_ipa_fold_scalars_dev(field_id, C.c_void_p(d_a_ptr), n, _capi.np_ptr(_fe(x)), _capi.np_ptr(_fe(y)),
                                                      _capi.FMT_CANONICAL, C.c_void_p(stream)))


def ipa_fold_bases(curve_id, d_bases_ptr, n, x, y, stream=0):
    _capi.check(_capi.lib().lurk_ipa_fold_bases_dev(curve_id, C.c_void_p(d_bases_ptr), n, _capi.np_ptr(_fe(x)), _capi.np_ptr(_fe(y)),
                                                    _capi.FMT_CANONICAL, C.c_void_p(stream)))


def ipa_prove(curve_id, ck, ck_c, d_a_ptr, d_b_ptr, log_n, challenge, stream=0):
    """InnerProductArgument::prove's rounds under the key of CommitmentKey `ck` (not consumed).  ck_c: (x, y) canonical ints.
    Returns (L points, R points, a_final, b_final); points are (x, y) tuples or None for the identity."""
    gc = np.concatenate([_fe(ck_c[0]), _fe(ck_c[1])])
    Ls = np.zeros(max(1, log_n) * 96, dtype=np.uint8)
    Rs = np.zeros(max(1, log_n) * 96, dtype=np.uint8)
    af, bf = np.zeros(32, dtype=np.uint8), np.zeros(32, dtype=np.uint8)
    errors = []
    cb = _callback(challenge, errors)
    rc = _capi.lib().lurk_ipa_prove_dev(curve_id, ck._ctx, _capi.np_ptr(gc), C.c_void_p(d_a_ptr), C.c_void_p(d_b_ptr), log_n, cb,
                                        None, _capi.np_ptr(Ls), _capi.np_ptr(Rs), _capi.np_ptr(af), _capi.np_ptr(bf), _capi.FMT_CANONICAL,
                                        C.c_void_p(stream))
    if errors:
        raise errors[0]
    _capi.check(rc)

    def pts(buf):
        out = []
        for i in range(log_n):
            b = buf[96 * i:96 * i + 96].tobytes()
            z = int.from_bytes(b[64:], "little")
            out.append((int.from_bytes(b[:32], "little"), int.from_bytes(b[32:64], "little")) if z else None)
        return out
    return pts(Ls), pts(Rs), int.from_bytes(af.tobytes(), "little"), int.from_bytes(bf.tobytes(), "little")


def hyperkzg_prove(curve_id, ck, d_poly_ptr, point, challenge, stream=0):
    """provider::hyperkzg::EvaluationEngine::prove.  ck: a CommitmentKey on the KZG key; point: ints.  challenge(round, message) -> int
    with round 0 = commitments, 1 = evaluations, 2 = witness commitments.  Returns (com points, v [3][l] ints, w points)."""
    l = len(point)
    pt = np.frombuffer(b"".join(int(x).to_bytes(32, "little") for x in point), dtype=np.uint8).copy()
    com = np.zeros(max(1, l - 1) * 96, dtype=np.uint8)
    w = np.zeros(3 * 96, dtype=np.uint8)
    v = np.zeros(3 * l * 32, dtype=np.uint8)
    errors = []
    cb = _callback(challenge, errors)
    rc = _capi.lib().lurk_hyperkzg_prove_dev(curve_id, ck._ctx, C.c_void_p(d_poly_ptr), _capi.np_ptr(pt), l, cb, None, _capi.np_ptr(com),
                                             _capi.np_ptr(w), _capi.np_ptr(v), _capi.FMT_CANONICAL, C.c_void_p(stream))
    if errors:
        raise errors[0]
    _capi.check(rc)

    def pts(buf, k):
        out = []
        for i in range(k):
            b = buf[96 * i:96 * i + 96].tobytes()
            out.append((int.from_bytes(b[:32], "little"), int.from_bytes(b[32:64], "little")) if int.from_bytes(b[64:], "little") else None)
        return out
    vi = _ints(v)
    return pts(com, l - 1), [vi[t * l:(t + 1) * l] for t in range(3)], pts(w, 3)



# ------------------------------------------------------------------------------------------------ RelaxedR1CSSNARK::prove, the GPU half
class DeviceCSR:
    """a CSR matrix resident on the GPU (row_ptr u64, col u32, val Montgomery field elements)"""

    def __init__(self, field_id, rows, row_ptr, col, val_canonical):
        import torch
        self.rows = rows
        self.rp = torch.from_numpy(np.ascontiguousarray(row_ptr, dtype=np.uint64).view(np.int64)).cuda()
        self.col = torch.from_numpy(np.ascontiguousarray(col, dtype=np.uint32).view(np.int32)).cuda()
        self.val = torch.from_numpy(np.ascontiguousarray(val_canonical, dtype=np.uint8).reshape(-1)).cuda()
        if self.val.numel():
            _capi.check(_capi.lib().lurk_convert_dev(field_id, C.c_void_p(self.val.data_ptr()), self.val.numel() // 32, _capi.FMT_MONTGOMERY,
                                                     C.c_void_p(self.val.data_ptr()), None))

    def mv(self, field_id, d_z_ptr, d_y_ptr):
        _capi.check(_capi.lib().lurk_spmv_csr_dev(field_id, C.c_void_p(self.rp.data_ptr()), C.c_void_p(self.col.data_ptr()), C.c_void_p(self.val.data_ptr()),
                                                  self.rows, C.c_void_p(d_z_ptr), C.c_void_p(d_y_ptr), None))


def padded_and_transposed(mats, n_w, num_vars, rows_pad):
    """host-side set-up (once per circuit shape): columns re-based onto the padded z = (W | 0.. | u | X | 0..) of length 2 num_vars, and the
    transposes (for compute_eval_table_sparse: sum_row eq(rx)[row] M[row][col]) as CSR over 2 num_vars rows.  mats: [(row_ptr, col, val bytes)]"""
    fwd, tr = [], []
    for rp, col, val in mats:
        rp = np.asarray(rp, dtype=np.uint64)
        col = np.asarray(col, dtype=np.int64)
        colm = np.where(col < n_w, col, num_vars + (col - n_w))
        val = np.ascontiguousarray(val, dtype=np.uint8).reshape(-1, 32)
        nrows = len(rp) - 1
        fwd.append((nrows, rp, colm.astype(np.uint32), val.reshape(-1)))
        row_of = np.repeat(np.arange(nrows, dtype=np.int64), np.diff(rp.astype(np.int64)))
        order = np.argsort(colm, kind="stable")
        trp = np.concatenate([[0], np.cumsum(np.bincount(colm, minlength=2 * num_vars))]).astype(np.uint64)
        tr.append((2 * num_vars, trp, row_of[order].astype(np.uint32), val[order].reshape(-1)))
    return fwd, tr


class RelaxedR1CSProver:
    """Control flow of Arecibo's spartan::snark::RelaxedR1CSSNARK::prove (reached from `compress`, reference src/proof/nova.rs:341-356) over the
    C-ABI primitives, every vector device-resident: multiply_vec (SpMV x3), EqPolynomial::evals, the outer (cubic) and inner (quadratic)
    sum-checks, compute_eval_table_sparse (transposed SpMV x3 + AXPY x2) and the evaluation claims.  The Fiat-Shamir transcript is a
    callable `challenge(label, data) -> int`; the polynomial-commitment openings (hyperkzg_prove / ipa_prove) are separate calls."""

    def __init__(self, field_id, mats, n_w, n_x):
        self.field = field_id
        self.p = int.from_bytes(field_modulus(field_id), "little")
        self.n_w, self.n_x = n_w, n_x
        self.rows = len(mats[0][0]) - 1
        self.log_rows = max(1, (self.rows - 1).bit_length())
        self.num_vars = 1 << max(1, (max(n_w, n_x + 1) - 1).bit_length())
        fwd, tr = padded_and_transposed(mats, n_w, self.num_vars, 1 << self.log_rows)
        self.M = [DeviceCSR(field_id, *m) for m in fwd]
        self.MT = [DeviceCSR(field_id, *m) for m in tr]

    def _mont(self, x):
        return _fe(int(x) * (1 << 256) % self.p)

    def _axpy(self, a, b, r, out):
        _capi.check(_capi.lib().lurk_axpy_dev(self.field, C.c_void_p(a.data_ptr()), C.c_void_p(b.data_ptr()), _capi.np_ptr(self._mont(r)), a.numel() // 32,
                                              C.c_void_p(out.data_ptr()), None))

    def pad_z(self, d_W, u, X):
        """(W | 0.. | u | X | 0..), Montgomery, 2 num_vars elements; d_W: device tensor of n_w Montgomery elements"""
        import torch
        z = torch.zeros(2 * self.num_vars * 32, dtype=torch.uint8, device="cuda")
        z[:self.n_w * 32] = d_W[:self.n_w * 32]
        tail = np.concatenate([self._mont(u)] + [self._mont(x) for x in X])
        z[self.num_vars * 32:self.num_vars * 32 + tail.size] = torch.from_numpy(tail).cuda()
        return z

    def prove(self, d_z, d_E, u, challenge, timings=None):
        """d_z: padded z (pad_z); d_E: device tensor of `rows` Montgomery elements.  Returns the transcript the verifier needs plus the points
        (rx, ry) at which E and W have to be opened."""
        import time
        import torch
        f, p, s, nv = self.field, self.p, self.log_rows, self.num_vars
        n_rows_pad = 1 << s
        t = time.perf_counter

        def mark(name, t0):
            if timings is not None:
                torch.cuda.synchronize()
                timings[name] = timings.get(name, 0.0) + (t() - t0) * 1e3

        t0 = t()
        Az, Bz, Cz = (torch.zeros(n_rows_pad * 32, dtype=torch.uint8, device="cuda") for _ in range(3))
        for M, y in zip(self.M, (Az, Bz, Cz)):
            M.mv(f, d_z.data_ptr(), y.data_ptr())
        E = torch.zeros(n_rows_pad * 32, dtype=torch.uint8, device="cuda")
        E[:self.rows * 32] = d_E[:self.rows * 32]
        uCzE = torch.empty_like(E)
        self._axpy(E, Cz, u, uCzE)
        mark("multiply_vec + u Cz + E", t0)
        t0 = t()
        tau = [challenge("tau", i) % p for i in range(s)]
        eq_tau = torch.empty(n_rows_pad * 32, dtype=torch.uint8, device="cuda")
        eq_evals(f, tau, eq_tau.data_ptr())
        mark("eq(tau)", t0)
        t0 = t()
        work = [eq_tau, Az.clone(), Bz.clone(), uCzE]
        outer_rounds, rx, fin = sumcheck_prove(f, CUBIC, [w.data_ptr() for w in work], s, 0,
                                               lambda rnd, msg: challenge("outer", (rnd, _ints(np.frombuffer(msg, dtype=np.uint8)))) % p)
        mark("outer sum-check", t0)
        t0 = t()
        eq_rx = torch.empty(n_rows_pad * 32, dtype=torch.uint8, device="cuda")
        eq_evals(f, rx, eq_rx.data_ptr())
        claims = (fin[1], fin[2], inner_product(f, Cz.data_ptr(), eq_rx.data_ptr(), n_rows_pad), inner_product(f, E.data_ptr(), eq_rx.data_ptr(), n_rows_pad))
        mark("claims at rx", t0)
        t0 = t()
        r = challenge("inner_r", claims) % p
        ys = [torch.empty(2 * nv * 32, dtype=torch.uint8, device="cuda") for _ in range(3)]
        for M, y in zip(self.MT, ys):
            M.mv(f, eq_rx.data_ptr(), y.data_ptr())
        abc = torch.empty_like(ys[0])
        self._axpy(ys[0], ys[1], r, abc)
        self._axpy(abc, ys[2], r * r % p, abc)
        mark("eval table (transposed SpMV)", t0)
        t0 = t()
        joint = (claims[0] + r * claims[1] + r * r * claims[2]) % p
        zc = d_z.clone()
        inner_rounds, ry, fin2 = sumcheck_prove(f, QUAD, [abc.data_ptr(), zc.data_ptr()], nv.bit_length(), joint,
                                                lambda rnd, msg: challenge("inner", (rnd, _ints(np.frombuffer(msg, dtype=np.uint8)))) % p)
        mark("inner sum-check", t0)
        t0 = t()
        eq_ry = torch.empty(nv * 32, dtype=torch.uint8, device="cuda")
        eq_evals(f, ry[1:], eq_ry.data_ptr())
        eval_W = inner_product(f, d_z.data_ptr(), eq_ry.data_ptr(), nv)
        mark("eval W", t0)
        return dict(outer_rounds=outer_rounds, inner_rounds=inner_rounds, claims=claims, eval_W=eval_W, rx=rx, ry=ry, E_padded=E)


# ------------------------------------------------------------------------------------------------ batch_eval_reduce + BatchedRelaxedR1CSSNARK
def _powers(x, n, p):
    out = [1]
    for _ in range(n - 1):
        out.append(out[-1] * x % p)
    return out[:n]


def _round_challenge(challenge, label, p):
    return lambda rnd, msg: challenge(label, (rnd, _ints(np.frombuffer(msg, dtype=np.uint8)))) % p


def batch_eval_prove(field_id, claims, challenge, open):
    """Arecibo's batch_eval_reduce (spartan/mod.rs) -- every evaluation claim of a proof reduced to one claim about one joint
    polynomial, so a circuit needs ONE polynomial-commitment opening.  claims: [(d_P, point, value)], d_P a device tensor of at least
    2^len(point) Montgomery elements (read, not modified), value = P(point).  With m_j = len(point_j), m = max m_j:
      sigma = challenge("batch_r", values); a batched quadratic sum-check over (copy of P_j, eq(point_j)), coefficients sigma^j, round
      challenges challenge("batch", (round, evals)) -> rho (m elements), left_j = P_j(rho[m - m_j:]);
      gamma = challenge("batch_g", left); P = sum_j gamma^j P_j (zero-extended to 2^m: lurk_poly_combine_dev);
      v = sum_j gamma^j L0_j left_j with L0_j = prod_{t < m - m_j} (1 - rho_t)  (= P(rho));  opening = open(P, rho, v).
    The verifier's joint commitment is sum_j gamma^j comm_j: zero-extension leaves a commitment unchanged."""
    import torch
    p = int.from_bytes(field_modulus(field_id), "little")
    ms = [len(pt) for _, pt, _ in claims]
    m = max(ms)
    values = [int(v) % p for _, _, v in claims]
    sigma = challenge("batch_r", values) % p
    work = []
    for (d_P, pt, _), mj in zip(claims, ms):
        P = d_P[:(1 << mj) * 32].clone()
        eq = torch.empty_like(P)
        eq_evals(field_id, [int(x) % p for x in pt], eq.data_ptr())
        work.append(([P.data_ptr(), eq.data_ptr()], mj, (P, eq)))
    rounds, rho, fin = sumcheck_prove_batch(field_id, QUAD, [(ptrs, mj) for ptrs, mj, _ in work], values, _powers(sigma, len(claims), p),
                                            _round_challenge(challenge, "batch", p))
    del work
    left = [f[0] for f in fin]
    gamma = challenge("batch_g", left) % p
    gp = _powers(gamma, len(claims), p)
    v = 0
    for g, mj, lj in zip(gp, ms, left):
        l0 = 1
        for t in range(m - mj):
            l0 = l0 * (1 - rho[t]) % p
        v = (v + g * l0 * lj) % p
    joint = torch.empty((1 << m) * 32, dtype=torch.uint8, device="cuda")
    poly_combine(field_id, [(d_P.data_ptr(), 1 << mj) for (d_P, _, _), mj in zip(claims, ms)], gp, joint.data_ptr(), 1 << m)
    opening = open(joint, rho, v)
    return dict(rounds=rounds, rho=rho, values=values, left=left, gamma=gamma, v=v, opening=opening)


def fold_running_inputs(prover, ctx):
    """(padded z, E, u, X) of a NovaFoldContext's running instance for `prover` (same R1CS shape), read where the fold keeps them:
    W and E stay on the device (LURK_FOLD_BUF_Z1 / E1); only u and X (a few elements) are copied to the host."""
    from .fold import device_tensor
    ctx.sync()                                       # the fold's streams are done with the running instance
    zp, zn = ctx.device_buffer(0, _capi.FOLD_BUF_Z1)
    ep, en = ctx.device_buffer(0, _capi.FOLD_BUF_E1)
    z1, e1 = device_tensor(zp, zn), device_tensor(ep, en)
    tail = z1[prover.n_w * 32:(prover.n_w + 1 + prover.n_x) * 32].clone()
    _capi.check(_capi.lib().lurk_convert_dev(prover.field, C.c_void_p(tail.data_ptr()), tail.numel() // 32, _capi.FMT_CANONICAL,
                                             C.c_void_p(tail.data_ptr()), None))
    ux = _ints(tail.cpu().numpy())
    return prover.pad_z(z1, ux[0], ux[1:]), e1, ux[0], ux[1:]


class BatchedRelaxedR1CSProver:
    """Control flow of Arecibo's spartan::batched::BatchedRelaxedR1CSSNARK::prove (SuperNova's `compress`, reference
    src/proof/supernova.rs:110,293-317): the running instances of ALL circuits of an NIVC proof in one argument.  One
    RelaxedR1CSProver per circuit supplies the device-resident matrices, their transposes and pad_z.  Instance i joins every batched
    sum-check late and uses the suffix of each shared challenge vector: r_x_i = r_x[s_max - s_i:], r_y_i = r_y[t_max - t_i:]."""

    def __init__(self, provers):
        self.provers = list(provers)
        self.field = self.provers[0].field
        self.p = self.provers[0].p
        if any(pr.field != self.field for pr in self.provers):
            raise ValueError("all instances of a batched proof live in one field")

    def prove(self, inputs, challenge, open=None, timings=None):
        """inputs: per instance (d_z, d_E, u, X) -- padded z (RelaxedR1CSProver.pad_z or fold_running_inputs) and `rows` Montgomery
        elements of E, device tensors.  Transcript (challenge(label, data) -> int):
          rho = challenge("outer_r", [(u_i, X_i)]); tau_t = challenge("tau", t), t < s_max; batched cubic sum-check of
          eq(tau_i) (Az_i Bz_i - (u_i Cz_i + E_i)), claims 0, coefficients rho^i, rounds challenge("outer", ...) -> r_x;
          claims_i = (Az_i, Bz_i, Cz_i, E_i) at r_x_i; r = challenge("inner_r", claims); batched quadratic sum-check of
          (A_i + r B_i + r^2 C_i)(r_x_i, .) z_i, claims Az + r Bz + r^2 Cz, coefficients (r^3)^i, rounds challenge("inner", ...) -> r_y;
          eval_W_i = W_i(r_y_i[1:]).
        Then, if `open` is given, batch_eval_prove over (W_i, r_y_i[1:], eval_W_i) for every i followed by (E_i, r_x_i, E_i(r_x_i))
        and the one opening open(d_P, point, value).  Returns the transcript; `eval_claims` are the 2k claims that were reduced."""
        import time
        import torch
        f, p, k = self.field, self.p, len(self.provers)
        t = time.perf_counter

        def mark(name, t0):
            if timings is not None:
                torch.cuda.synchronize()
                timings[name] = timings.get(name, 0.0) + (t() - t0) * 1e3

        def dev(n):
            return torch.zeros(n * 32, dtype=torch.uint8, device="cuda")
        s = [pr.log_rows for pr in self.provers]
        tv = [pr.num_vars.bit_length() for pr in self.provers]         # log2(2 num_vars)
        s_max, t_max = max(s), max(tv)
        t0 = t()
        prods, Es = [], []
        for pr, (d_z, d_E, u, _) in zip(self.provers, inputs):
            Az, Bz, Cz = dev(1 << pr.log_rows), dev(1 << pr.log_rows), dev(1 << pr.log_rows)
            for M, y in zip(pr.M, (Az, Bz, Cz)):
                M.mv(f, d_z.data_ptr(), y.data_ptr())
            E = dev(1 << pr.log_rows)
            E[:pr.rows * 32] = d_E[:pr.rows * 32]
            uCzE = torch.empty_like(E)
            pr._axpy(E, Cz, u, uCzE)
            prods.append((Az, Bz, Cz, uCzE))
            Es.append(E)
        mark("multiply_vec + u Cz + E", t0)
        t0 = t()
        rho = challenge("outer_r", [(int(u) % p, [int(x) % p for x in X]) for _, _, u, X in inputs]) % p
        tau = [challenge("tau", i) % p for i in range(s_max)]
        work = []
        for si, (Az, Bz, _, uCzE) in zip(s, prods):
            eq_tau = torch.empty_like(Az)
            eq_evals(f, tau[s_max - si:], eq_tau.data_ptr())
            work.append(([eq_tau, Az.clone(), Bz.clone(), uCzE], si))
        outer_rounds, rx, fin = sumcheck_prove_batch(f, CUBIC, [([x.data_ptr() for x in w], si) for w, si in work], [0] * k,
                                                     _powers(rho, k, p), _round_challenge(challenge, "outer", p))
        del work
        mark("outer sum-check", t0)
        t0 = t()
        eq_rx, claims = [], []
        for i, (si, (_, _, Cz, _), E) in enumerate(zip(s, prods, Es)):
            e = torch.empty_like(E)
            eq_evals(f, rx[s_max - si:], e.data_ptr())
            eq_rx.append(e)
            claims.append((fin[i][1], fin[i][2], inner_product(f, Cz.data_ptr(), e.data_ptr(), 1 << si), inner_product(f, E.data_ptr(), e.data_ptr(), 1 << si)))
        del prods
        mark("claims at rx", t0)
        t0 = t()
        r = challenge("inner_r", claims) % p
        abcs = []
        for pr, e in zip(self.provers, eq_rx):
            ys = [torch.empty(2 * pr.num_vars * 32, dtype=torch.uint8, device="cuda") for _ in range(3)]
            for M, y in zip(pr.MT, ys):
                M.mv(f, e.data_ptr(), y.data_ptr())
            abc = torch.empty_like(ys[0])
            pr._axpy(ys[0], ys[1], r, abc)
            pr._axpy(abc, ys[2], r * r % p, abc)
            abcs.append(abc)
        del eq_rx
        mark("eval table (transposed SpMV)", t0)
        t0 = t()
        joints = [(c[0] + r * c[1] + r * r * c[2]) % p for c in claims]
        zcs = [d_z[:2 * pr.num_vars * 32].clone() for pr, (d_z, _, _, _) in zip(self.provers, inputs)]
        inner_rounds, ry, _ = sumcheck_prove_batch(f, QUAD, [([abc.data_ptr(), zc.data_ptr()], ti) for abc, zc, ti in zip(abcs, zcs, tv)], joints,
                                                   _powers(r * r * r % p, k, p), _round_challenge(challenge, "inner", p))
        del abcs, zcs
        mark("inner sum-check", t0)
        t0 = t()
        eval_W = []
        for pr, ti, (d_z, _, _, _) in zip(self.provers, tv, inputs):
            eq_ry = torch.empty(pr.num_vars * 32, dtype=torch.uint8, device="cuda")
            eq_evals(f, ry[t_max - ti + 1:], eq_ry.data_ptr())
            eval_W.append(inner_product(f, d_z.data_ptr(), eq_ry.data_ptr(), pr.num_vars))
        mark("eval W", t0)
        eval_claims = ([(d_z, ry[t_max - ti + 1:], ew) for (d_z, _, _, _), ti, ew in zip(inputs, tv, eval_W)]
                       + [(E, rx[s_max - si:], c[3]) for E, si, c in zip(Es, s, claims)])
        out = dict(outer_rounds=outer_rounds, inner_rounds=inner_rounds, claims=claims, eval_W=eval_W, rx=rx, ry=ry, E_padded=Es,
                   eval_claims=eval_claims)
        if open is not None:
            t0 = t()
            out["batch"] = batch_eval_prove(f, eval_claims, challenge, open)
            mark("batch_eval_reduce + opening", t0)
        return out
