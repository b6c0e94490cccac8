#!/usr/bin/env python3
"""bench.py -- Lurk reduction iterations proved per second on the GPU hot path (BASELINE.json metric).

Workload `fib` (default): the per-fold GPU work of `benches/fibonacci.rs` at rc = 100 (Nova IVC, BN254 / Grumpkin cycle
as the reference bench really runs -- SURVEY.md D1), driven ONLY through the fold context of the C ABI
(lurk_fold_ctx_*, include/lurk_b200.h), i.e. what RecursiveSNARK::prove_step does with the step circuit's witness inside
Arecibo's NIFS::prove (SURVEY.md Appendix B), on synthetic inputs of the real shapes:
    stage A  H2D of the step's inputs (slot preimages, LEM-body aux, public IO);  1400 Hash4 + 600 Hash8 + 100 Commitment
             Poseidon slot witnesses + 300 bit decompositions written in place into W2 (src/lem/eval.rs:1960-1964);
             comm_W2 = commit(W2), |W| = rc * 9119 = 911 900 (eval.rs:1966);  A z2, B z2, C z2
    stage B  A z1, B z1, C z1;  cross term T over rc * 11141 = 1 114 100 rows (eval.rs:1967);  comm_T = commit(T);
             Poseidon-sponge random oracle -> r;  (W, u, X) += r (W2, 1, X2), E += r T;  comm_W += r comm_W2, comm_E += r comm_T
    + the same fold of the ~10^4-constraint secondary circuit on Grumpkin (second context)
A "step" is one fold = rc iterations.  The R1CS is synthetic but SATISFIABLE by construction (per frame 1311 product rows
that define the LEM-body aux from slot-witness columns, 9830 linear rows), so the folded running instance is CHECKED
before timing: relaxed R1CS residual = 0 and commit(W), commit(E) equal the folded commitments (on the device), and one
full-size fold's comm_W2, comm_T and challenge are compared with the CPU oracle.  Not included (CPU work of the
reference that is out of scope, SURVEY.md 8(a) a7): LEM synthesis of the body aux, Nova's augmented-circuit synthesis.

N > 1 (torchrun, one process per GPU): frames, witness, matrix rows and the commitment key are split by frame across ranks;
the only exchange is the two partial commitments per step, written peer-to-peer into every rank's exchange buffer over
NVLink by the challenge kernel itself (no NCCL call, no host hop on the chain).  --scaling weak: rc = 100 * N (the
reference layout of a larger step circuit); --scaling strong: ONE rc = 100 fold, its 2^21-point key split N ways.

`--impl reference` times the CPU restatement of the same step (oracle/, all host threads): the reference's own prover
is Rust and cannot be built in this image (DESIGN.md).
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

RC = 100                      # frames per step (benches/fibonacci.rs default LURK_RC=100)
AUX_PER_FRAME = 9119          # src/lem/eval.rs:1966
CONS_PER_FRAME = 11141        # src/lem/eval.rs:1967
SLOTS = [(4, 14), (8, 6), (3, 1)]   # (arity, slots per frame); hash6 has no slots (eval.rs:1960-1964)
BITDECOMP_PER_FRAME = 3
SLOT_ELEMS = 7808             # 14*293 + 6*396 + 268 + 3*354 (multiframe.rs:991-1016)
GLUE_PER_FRAME = AUX_PER_FRAME - SLOT_ELEMS     # 1311 LEM-body aux
SECONDARY_N = 10_000          # secondary-circuit witness / constraint count (order of magnitude, SURVEY.md 8(a) a10)
CURVE, CURVE2 = 0, 1          # BN254 G1 primary (witness field Fr), Grumpkin secondary (witness field Fq)
LIVE_SLOT_FRACTION = 0.25     # most slots of a frame are dummies (multiframe.rs:553-577)
PP_DIGEST = 0x2c5d1f0a9b8e7d6c5b4a39281706f5e4d3c2b1a0918273645546372819
P_FR = 0x30644e72e131a029b85045b68181585d2833e84879b9709143e1f593f0000001
P_FQ = 0x30644e72e131a029b85045b68181585d97816a916871ca8d3c208c16d87cfd47
METRIC = "Lurk iterations proved/sec (fib rc=100, Nova IVC)"


def rand_elements(rng, count, shape="uniform"):
    raw = rng.integers(0, 256, size=(count, 32), dtype=np.uint8)
    raw[:, 31] &= 0x1f                                   # < 2^253 < p for every field used here
    if shape == "witness":                                # 40% 0/1, 10% < 2^16, 50% uniform (SURVEY.md 8(d))
        u = rng.random(count)
        small = u < 0.4
        raw[small] = 0
        raw[small, 0] = rng.integers(0, 2, size=int(small.sum()), dtype=np.uint8)
        mid = (u >= 0.4) & (u < 0.5)
        raw[mid, 2:] = 0
    return raw.reshape(-1)


def small_vals(rng, n):
    val = np.zeros((n, 32), dtype=np.uint8)
    val[:, 0] = rng.integers(1, 8, size=n, dtype=np.uint8)
    return val.reshape(-1)


def step_circuit(seed, frames, slot_elems=SLOT_ELEMS, glue=GLUE_PER_FRAME, cons=CONS_PER_FRAME, n_x=2, linear_fraction=0.02, bits=0):
    """Synthetic R1CS in the shape of the Lurk step circuit, satisfiable by construction AND with a dense cross term (as the
    real circuit's: every constraint is a genuine product).  Frame = [slot_elems free columns | glue defined columns | bits
    boolean columns].  Per frame: `glue` defining rows (a_k . slots)(b_k . slots) = glue_k -- the LEM-body aux stand-in --,
    cons - glue further rows that re-state a definition k = row mod glue with other coefficients, (l a_k . slots)(m b_k . slots)
    = l m glue_k, except a small fraction of linear rows (a . z) u = (a . z) that also touch the public IO (their cross term
    vanishes identically), and one booleanity row b * b = b per boolean column (the SHA-256 gadget's witness, config 4).
    Columns: frame-major W, then u, then X.  Values are canonical small integers.
    Returns [(row_ptr, col, val)] x 3, n_w, rows, the global row index of every defining row."""
    rng = np.random.default_rng(seed)
    per = slot_elems + glue + bits
    rows_pf = cons + bits
    n_w, rows = frames * per, frames * rows_pf
    # ---- the definitions of one frame layout (shared by all frames up to the column base)
    na = rng.integers(1, 4, size=glue)                       # non-zeros of a_k: 1..3
    nb = rng.integers(1, 3, size=glue)                       # non-zeros of b_k: 1..2
    a_ptr = np.concatenate([[0], np.cumsum(na)])
    b_ptr = np.concatenate([[0], np.cumsum(nb)])
    a_col = rng.integers(0, slot_elems, size=int(a_ptr[-1]))
    b_col = rng.integers(0, slot_elems, size=int(b_ptr[-1]))
    a_cf = rng.integers(1, 4, size=int(a_ptr[-1]))
    b_cf = rng.integers(1, 4, size=int(b_ptr[-1]))
    # ---- rows of one frame: [cons product / linear rows | bits booleanity rows]
    local = np.arange(rows_pf)
    is_bool = local >= cons
    k = np.where(is_bool, 0, local % glue)
    is_lin = (local >= glue) & ~is_bool & (rng.random(rows_pf) < linear_fraction)
    own = is_lin | is_bool                                     # rows with their own entries instead of a definition's
    lam = np.where(local < glue, 1, rng.integers(1, 3, size=rows_pf))
    mu = np.where(local < glue, 1, rng.integers(1, 3, size=rows_pf))
    bit_col = slot_elems + glue + (local - cons)               # valid where is_bool

    def expand(ptr, col, cf, scale, own_cols, own_cf, own_cnt):
        """per-frame CSR of rows taking definition k's entries scaled, or the row's own entries (first own_cnt of them)"""
        cnt = np.where(own, own_cnt, ptr[k + 1] - ptr[k])
        rp = np.concatenate([[0], np.cumsum(cnt)])
        cols = np.empty(int(rp[-1]), dtype=np.int64)
        vals = np.empty(int(rp[-1]), dtype=np.int64)
        r_of = np.repeat(local, cnt)
        within = np.arange(int(rp[-1])) - rp[r_of]
        d = ~own[r_of]
        src = ptr[k[r_of[d]]] + within[d]
        cols[d] = col[src]
        vals[d] = cf[src] * scale[r_of[d]]
        cols[~d] = own_cols[r_of[~d], within[~d]]
        vals[~d] = own_cf[r_of[~d], within[~d]]
        return rp, cols, vals

    U = -100                                                   # marker of the u column; -1 - j marks public IO j
    # A: linear rows = two W columns of the frame + one public-IO column; boolean rows = the bit column
    lin_cols = np.stack([rng.integers(0, per, size=rows_pf), rng.integers(0, per, size=rows_pf), -1 - rng.integers(0, n_x, size=rows_pf)], axis=1)
    lin_cf = rng.integers(1, 4, size=(rows_pf, 3))
    a_own_cols = np.where(is_bool[:, None], bit_col[:, None], lin_cols)
    a_own_cf = np.where(is_bool[:, None], 1, lin_cf)
    fa = expand(a_ptr, a_col, a_cf, lam, a_own_cols, a_own_cf, np.where(is_bool, 1, 3))
    # B: linear rows = u; boolean rows = the bit column
    b_own_cols = np.where(is_bool, bit_col, U)[:, None]
    fb = expand(b_ptr, b_col, b_cf, mu, b_own_cols, np.ones((rows_pf, 1), dtype=np.int64), np.ones(rows_pf, dtype=np.int64))
    # C: defining / restating rows -> lam * mu at the glue column; linear rows -> their A row; boolean rows -> the bit column
    c_ptr = np.arange(glue + 1)
    fc = expand(c_ptr, slot_elems + np.arange(glue), np.ones(glue, dtype=np.int64), lam * mu, a_own_cols, a_own_cf, np.where(is_bool, 1, 3))

    def tile(frame_csr):
        rp, cols, vals = frame_csr
        nnz = int(rp[-1])
        all_rp = (np.arange(frames, dtype=np.int64)[:, None] * nnz + rp[None, :-1]).reshape(-1)
        all_rp = np.concatenate([all_rp, [frames * nnz]]).astype(np.uint64)
        base = np.arange(frames, dtype=np.int64)[:, None] * per
        c = np.where(cols[None, :] >= 0, base + cols[None, :], np.where(cols[None, :] == U, n_w, n_w + 1 + (-1 - cols[None, :])))
        v = np.zeros((frames * nnz, 32), dtype=np.uint8)
        v[:, 0] = np.tile(vals, frames).astype(np.uint8)
        return all_rp, c.reshape(-1).astype(np.uint32), v.reshape(-1)

    prod_rows = (np.arange(frames, dtype=np.int64)[:, None] * rows_pf + np.arange(glue)[None, :]).reshape(-1)
    return [tile(fa), tile(fb), tile(fc)], n_w, rows, prod_rows


def slot_offsets(frames, per, slots, bd_per_frame, field=0):
    """element offset of every slot block inside W, in the reference's frame layout (multiframe.rs:635-712): per frame
    [slot blocks in slot order | body aux ...]; returns ([(arity, offsets)], slot elements per frame)"""
    import lurk_beta_b200 as L
    lib = L._capi.lib()
    out, cur = [], 0
    f = np.arange(frames, dtype=np.uint64)[:, None] * per
    for arity, per_frame in slots:
        blk = lib.lurk_poseidon_witness_block(field, arity)
        out.append((arity, per_frame, (f + cur + np.arange(per_frame, dtype=np.uint64)[None, :] * blk).reshape(-1)))
        cur += per_frame * blk
    if bd_per_frame:
        blk = lib.lurk_bitdecomp_witness_block(field)
        out.append((0, bd_per_frame, (f + cur + np.arange(bd_per_frame, dtype=np.uint64)[None, :] * blk).reshape(-1)))
        cur += bd_per_frame * blk
    return out, cur


def to_mont(buf, p):
    """canonical 32-byte elements -> Montgomery bytes (host, setup only)"""
    b = np.ascontiguousarray(buf, dtype=np.uint8).tobytes()
    R = 1 << 256
    return np.frombuffer(b"".join((int.from_bytes(b[i:i + 32], "little") * R % p).to_bytes(32, "little") for i in range(0, len(b), 32)),
                         dtype=np.uint8).copy()


def workload_config(world, scaling, workload="fib", rc=RC):
    frames = rc * world if scaling == "weak" else rc
    cfg = {"workload": "fib rc=100 Nova IVC fold step on BN254/Grumpkin (benches/fibonacci.rs, configs[0]/metric config)",
           "composed": "per fold, through lurk_fold_ctx_*: H2D of slot preimages + LEM-body aux; 2100 Poseidon slot witnesses + 300 bit-decomps "
                       "per 100 frames; commit(W) 911900 terms; cross term over 1114100 rows (A z, B z, C z of the running instance kept current by "
                       "the fold); commit(T); Poseidon-sponge RO challenge; fold of (W,u,X), E and both commitments; the same fold of a "
                       "10^4-constraint secondary circuit on Grumpkin. LEM synthesis / augmented-circuit synthesis / reference Rust prover not included",
           "frames_per_step": frames, "scaling": scaling, "live_slot_fraction": LIVE_SLOT_FRACTION,
           "commitment_key": "2^21 synthetic BN254 G1 points per 100 frames ([i+1]G), sharded by frame; fixed-base window tables built once",
           "l2": "inputs per step (128 MiB key, 1.7 GB window table, 64 MiB of vectors, 140 MiB CSR) exceed the 126 MB L2",
           "parallelism": f"frames/bases sharded over {world} GPU(s); partial commitments exchanged through NVLink peer memory inside the challenge kernel"}
    if workload == "sha256_ivc":
        cfg["workload"] = (f"examples/sha256_ivc.rs shape (configs[3]): rc={rc}, every frame = Lurk frame + inlined SHA-256 gadget (45000 boolean aux "
                           "and booleanity constraints); |W| = rc * 54119, rows = rc * 56141; Nova IVC on BN254/Grumpkin")
    elif workload == "trie_nivc":
        cfg["workload"] = (f"benches/trie_nivc.rs shape (configs[4]): SuperNova NIVC, Lurk step circuit rc={rc} + trie-lookup coprocessor circuit "
                           "(85 arity-8 Poseidon witnesses, src/coprocessor/trie/mod.rs:592-640) + secondary circuit; one fold of each per step")
    return cfg


class ClockSampler:
    """samples SM clock and throttle reasons through NVML every few milliseconds during the timed region"""

    def __init__(self, index):
        self.index, self.sm, self.max_sm, self.reasons = index, [], None, set()
        self._stop = threading.Event()
        self._thread = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            ids = [int(x) for x in vis.split(",") if x.strip().isdigit()]
            phys = ids[self.index] if self.index < len(ids) else self.index
            h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            names = {"hw_slowdown": getattr(pynvml, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                     "hw_thermal_slowdown": getattr(pynvml, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                     "sw_thermal_slowdown": getattr(pynvml, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                     "sw_power_cap": getattr(pynvml, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}

            def loop():
                while not self._stop.is_set():
                    try:
                        self.sm.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                        mask = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                        self.reasons |= {k for k, bit in names.items() if mask & bit}
                    except Exception:
                        pass
                    time.sleep(0.004)
            self._thread = threading.Thread(target=loop, daemon=True)
            self._thread.start()
        except Exception:
            self._thread = None

    def stop(self):
        self._stop.set()
        if self._thread:
            self._thread.join(timeout=1.0)
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_sm, "reasons": sorted(self.reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------- GPU arm
# circuit shapes: (slots per frame, bit decompositions per frame, free host columns when there are no slots, glue, boolean
# columns, product/linear constraints) -- frame = [slot blocks | glue | bits]
LURK_FRAME = dict(slots=SLOTS, bd=BITDECOMP_PER_FRAME, free=0, glue=GLUE_PER_FRAME, bits=0, cons=CONS_PER_FRAME)
SECONDARY = dict(slots=[], bd=0, free=SECONDARY_N - 1500, glue=1500, bits=0, cons=SECONDARY_N)
# examples/sha256_ivc.rs (config 4): the SHA-256 gadget is inlined in every frame of the step circuit (src/coprocessor/sha256.rs:27-64):
# ~45 k boolean aux and as many constraints per frame on top of the Lurk frame, rc = 10 (examples/sha256_ivc.rs:20)
SHA256_FRAME = dict(slots=SLOTS, bd=BITDECOMP_PER_FRAME, free=0, glue=GLUE_PER_FRAME, bits=45_000, cons=CONS_PER_FRAME)
# trie lookup coprocessor circuit (config 5; src/coprocessor/trie/mod.rs:592-640): 85 arity-8 Poseidon witnesses + path glue
TRIE_LOOKUP = dict(slots=[(8, 85)], bd=0, free=0, glue=2_000, bits=0, cons=40_000)


class Instance:
    """one circuit of the proof = one fold context, with the synthetic inputs of two distinct fresh instances in its pinned buffers"""

    def __init__(self, torch, L, curve, shape, frames, ck_w, ck_t, world, rank, seed, live, x2, latency_sms=0):
        self.torch, self.L, self.curve, self.frames = torch, L, curve, frames
        self.p_w, self.p_base = (P_FR, P_FQ) if curve == CURVE else (P_FQ, P_FR)
        self.field = 0 if curve == CURVE else 1
        M = L.FMT_MONTGOMERY
        layout, slot_elems = slot_offsets(frames, 0, shape["slots"], shape["bd"], self.field)     # first pass: sizes only
        self.slot_elems = slot_elems or shape["free"]
        self.glue, self.bits = shape["glue"], shape["bits"]
        self.per = self.slot_elems + self.glue + self.bits
        layout, _ = slot_offsets(frames, self.per, shape["slots"], shape["bd"], self.field)
        self.mats, self.nW, self.nT, self.prod_rows = step_circuit(seed, frames, slot_elems=self.slot_elems, glue=self.glue, cons=shape["cons"],
                                                                   bits=self.bits)
        self.ctx = L.NovaFoldContext(curve, ck_w, self.nW, 2, self.mats, depth=2, fmt=L.FMT_CANONICAL, ck_t=ck_t, world=world, rank=rank,
                                     latency_sms=latency_sms)
        self.batch = [(arity, per_frame, self.ctx.add_slot_batch(arity, offs)) for arity, per_frame, offs in layout]
        self.has_slots = bool(self.batch)
        if self.has_slots:
            self.ctx.set_spans([(self.slot_elems, self.glue + self.bits, self.per, frames)])
        else:
            self.ctx.set_spans([(0, self.nW, self.nW, 1)])          # the whole witness comes from the host
        self.x2 = x2
        rng = np.random.default_rng(seed + 1)
        one = to_mont(FoldStepGPU._pack([1]), self.p_w)
        # Every input is handed over in Montgomery form (the in-memory form of halo2curves' field types); random bytes < p are
        # valid Montgomery representatives of uniformly random elements.  The two fresh-instance buffers get DIFFERENT inputs:
        # folding the same instance over and over would make every cross term vanish identically.
        for b in range(2):
            for arity, per_frame, idx in self.batch:
                n = frames * per_frame
                if arity:
                    x = rand_elements(rng, n * arity).reshape(n, arity * 32)
                    x[rng.random(n) >= live] = 0
                    self.ctx.host_buffer(b, idx)[:] = x.reshape(-1)
                else:
                    self.ctx.host_buffer(b, idx)[:] = rand_elements(rng, n, "witness")
            host = self.ctx.host_buffer(b, L._capi.FOLD_BUF_GLUE)
            rows = host.reshape(frames, -1)                          # per frame: [glue | bits] or [free | glue | bits]
            row_elems = rows.shape[1] // 32
            if not self.has_slots:
                rows[:, :self.slot_elems * 32] = rand_elements(rng, frames * self.slot_elems, "witness").reshape(frames, -1)
            if self.bits:
                bitv = np.zeros((frames, self.bits, 32), dtype=np.uint8)
                bitv[rng.random((frames, self.bits)) < 0.5] = one
                rows[:, (row_elems - self.bits) * 32:] = bitv.reshape(frames, -1)
            self.ctx.host_buffer(b, L._capi.FOLD_BUF_X2)[:] = to_mont(FoldStepGPU._pack(x2), self.p_w)
            ro = np.zeros((24, 32), dtype=np.uint8)
            for pos, v in ((0, PP_DIGEST), (4, x2[0]), (5, x2[1])):
                ro[pos] = FoldStepGPU._pack([v])
            self.ctx.host_buffer(b, L._capi.FOLD_BUF_RO)[:] = to_mont(ro.reshape(-1), self.p_base)
            self._derive_glue(b)
        self.h2d_bytes = sum(self.ctx.host_buffer(0, w).size for w in [i for _, _, i in self.batch] + [-1, -2, -3])

    def _derive_glue(self, b):
        """setup: make the fresh instance satisfy the circuit -- glue_g = (A_g . z)(B_g . z) for the defining rows, computed with
        the library's own SpMV / cross-term kernels on the device from the slot columns the slot kernels produce"""
        t, L, ctx = self.torch, self.L, self.ctx
        lib = L._capi.lib()
        M = L.FMT_MONTGOMERY
        ctx.stage_a(b, fmt=M)          # with the glue still zero: fills the slot columns of W2 / uploads the free columns
        ctx.sync()
        z2 = ctx.device_view(b, L._capi.FOLD_BUF_W2)
        dev = lambda a: t.from_numpy(np.ascontiguousarray(a)).cuda()
        out = []
        for rp, col, val in self.mats[:2]:
            y = t.empty(self.nT * 32, dtype=t.uint8, device="cuda")
            d = (dev(rp), dev(col), dev(to_mont_small(val, self.p_w)))
            L._capi.check(lib.lurk_spmv_csr_dev(self.field, d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), self.nT, z2.data_ptr(), y.data_ptr(), None))
            out.append(y)
        zero = t.zeros(self.nT * 32, dtype=t.uint8, device="cuda")
        prod = t.empty(self.nT * 32, dtype=t.uint8, device="cuda")
        z32 = np.zeros(32, dtype=np.uint8)
        L._capi.check(lib.lurk_cross_term_dev(self.field, out[0].data_ptr(), zero.data_ptr(), zero.data_ptr(), zero.data_ptr(), out[1].data_ptr(),
                                              zero.data_ptr(), L._capi.np_ptr(z32), L._capi.np_ptr(z32), self.nT, prod.data_ptr(), None))
        t.cuda.synchronize()
        glue = prod.view(self.nT, 32)[dev(self.prod_rows.astype(np.int64))].cpu().numpy().reshape(self.frames, self.glue * 32)
        rows = ctx.host_buffer(b, L._capi.FOLD_BUF_GLUE).reshape(self.frames, -1)
        g0 = 0 if self.has_slots else self.slot_elems
        rows[:, g0 * 32:(g0 + self.glue) * 32] = glue
        del z2


class FoldStepGPU:
    """one rank's share of the fold step of a workload, driven through the C-ABI fold context"""

    def __init__(self, rank, world, scaling="weak", latency_sms=0, seed=0x6c75726b, workload="fib", rc=None, key="synthetic"):
        import torch
        import lurk_beta_b200 as L
        self.torch, self.L = torch, L
        self.rank, self.world, self.workload = rank, world, workload
        M = L.FMT_MONTGOMERY
        shape = SHA256_FRAME if workload == "sha256_ivc" else LURK_FRAME
        self.rc = rc or {"fib": RC, "sha256_ivc": 10, "trie_nivc": 400}[workload]
        total_frames = self.rc * world if scaling == "weak" else self.rc
        f0, f1 = (total_frames * rank) // world, (total_frames * (rank + 1)) // world
        self.frames = f1 - f0
        per = SLOT_ELEMS + shape["glue"] + shape["bits"]
        rows_pf = shape["cons"] + shape["bits"]
        nW, nT = self.frames * per, self.frames * rows_pf
        # ---- commitment key: this rank's slices of the global key [i+1]G in the reference's layout (W index = frame * per + j,
        # T / E index = frame * rows_per_frame + j).  One resident power-of-two key serves both when nothing is sharded.
        self.key, self.ck_generate_ms = key, None
        if key == "from_label":
            # the reference's own key distribution (N3): DlogGroup::from_label(b"ck", n) generated on the GPU into device memory
            t0 = time.perf_counter()
            if world == 1:
                n_key = L.ck_size(nT, nW, 1 << 14)
                self.ck_w = self.ck_t = L.CommitmentKey.setup(CURVE, b"ck", n_key)
            else:
                self.ck_w = L.CommitmentKey.setup(CURVE, b"ck", nW, first=f0 * per)
                self.ck_t = L.CommitmentKey.setup(CURVE, b"ck", nT, first=f0 * rows_pf)
            torch.cuda.synchronize()
            self.ck_generate_ms = (time.perf_counter() - t0) * 1e3
        elif world == 1:
            n_key = 1 << max(14, (max(nW, nT) - 1).bit_length())
            self.ck_w = self.ck_t = L.CommitmentKey(CURVE, L.synthetic_bases(CURVE, n_key, fmt=M), fmt=M)
        else:
            self.ck_w = L.CommitmentKey(CURVE, L.synthetic_bases(CURVE, nW, start=f0 * per, fmt=M), fmt=M)
            self.ck_t = L.CommitmentKey(CURVE, L.synthetic_bases(CURVE, nT, start=f0 * rows_pf, fmt=M), fmt=M)
        common = np.random.default_rng(seed + 99)                 # X / RO constants are identical on every rank (the challenge must agree)
        mk_x = lambda: [int(common.integers(1, 2**62)) * int(common.integers(1, 2**62)) for _ in range(2)]
        self.inst = [Instance(torch, L, CURVE, shape, self.frames, self.ck_w, self.ck_t, world, rank, seed + 1000 * rank, LIVE_SLOT_FRACTION, mk_x(),
                              latency_sms)]
        self.names = ["primary"]
        if workload == "trie_nivc":
            # the coprocessor circuit is small: replicated on every rank (world = 1 context), one lookup per Lurk step
            ck = self.ck_w if world == 1 else L.CommitmentKey(CURVE, L.synthetic_bases(CURVE, 1 << 17, fmt=M), fmt=M)
            self.ck_trie = ck
            self.inst.append(Instance(torch, L, CURVE, TRIE_LOOKUP, 1, ck, ck, 1, 0, seed + 5, 1.0, mk_x()))
            self.names.append("trie")
        # the secondary circuit of the cycle (Grumpkin): whole witness from the host, replicated on every rank
        self.ck2 = L.CommitmentKey(CURVE2, L.synthetic_bases(CURVE2, 1 << 14, fmt=M), fmt=M)
        if not os.environ.get("LURK_BENCH_NO_SECONDARY"):        # measurement aid (the chain of the primary circuit alone)
            self.inst.append(Instance(torch, L, CURVE2, SECONDARY, 1, self.ck2, self.ck2, 1, 0, seed + 7, 1.0, mk_x()))
            self.names.append("secondary")
        self.ctx = self.inst[0].ctx
        self.nW, self.nT, self.X2 = self.inst[0].nW, self.inst[0].nT, self.inst[0].x2
        self.h2d_bytes = sum(i.h2d_bytes for i in self.inst)
        self.d2h_bytes = 448 * len(self.inst)              # the result records
        self.step_index = 0
        self.started = False
        torch.cuda.synchronize()

    @staticmethod
    def _pack(vals):
        return np.frombuffer(b"".join(int(v).to_bytes(32, "little") for v in vals), dtype=np.uint8).copy()

    # ------------------------------------------------------------------------------------------ the step loop
    def start(self, staged):
        """RecursiveSNARK::new on buffer 0, stage A of the first fold on buffer 1"""
        M = self.L.FMT_MONTGOMERY
        for i in self.inst:
            i.ctx.stage_a(0, resident=not staged, fmt=M)
            i.ctx.init_running(0)
            i.ctx.stage_a(1, resident=not staged, fmt=M)
        for i in self.inst:
            i.ctx.collect(0)
        self.step_index = 1
        self.uncollected = None
        self.started = True

    def step(self, staged):
        """one fold of every circuit: enqueue stage B of step i, collect step i-1's records, enqueue stage A of step i+1 into the
        freed buffers"""
        k = self.step_index
        b = k & 1
        M = self.L.FMT_MONTGOMERY
        for i in self.inst:
            i.ctx.stage_b_launch(b)
        if self.uncollected is not None:
            self.last = [i.ctx.collect(self.uncollected) for i in self.inst]
        self.uncollected = b
        for i in self.inst:
            i.ctx.stage_a(b ^ 1, resident=not staged, fmt=M)
        self.step_index = k + 1

    def drain(self):
        """collect the last fold (the prefetched stage A of the step after it stays un-folded: it is extra work inside the region)"""
        if self.uncollected is not None:
            self.last = [i.ctx.collect(self.uncollected) for i in self.inst]
            self.uncollected = None
        for i in self.inst:
            i.ctx.sync()


def to_mont_small(val, p):
    """coefficients are small integers 1..7: Montgomery form through a table"""
    R = 1 << 256
    table = np.stack([np.frombuffer((k * R % p).to_bytes(32, "little"), dtype=np.uint8) for k in range(8)])
    return table[np.ascontiguousarray(val, dtype=np.uint8).reshape(-1, 32)[:, 0]].reshape(-1)


def verify_full_size(wl, rank):
    """outside the timed region: (1) the device-side relaxed-R1CS check of every running instance after real folds, on every rank
    (collective when the key is sharded); (2) rank 0 of an unsharded run: one full-size fold against the CPU oracle."""
    out = {"relaxed_r1cs_bad_rows": 0, "folded_commitments_open": True}
    for i in wl.inst:
        bad, okw, oke = i.ctx.check_running()
        out["relaxed_r1cs_bad_rows"] += int(bad)
        out["folded_commitments_open"] = bool(out["folded_commitments_open"] and okw and oke)
    if wl.world == 1 and rank == 0 and max(wl.nW, wl.nT) <= 5_000_000:
        from oracle import capi as oracle, spec, nifs   # checker only
        L = wl.L
        th = host_threads()
        rec = wl.last[0]
        ctx = wl.ctx
        b = (wl.step_index - 1) & 1
        W2 = ctx.read_device(b, L._capi.FOLD_BUF_W2)[:wl.nW * 32]
        T = ctx.read_device(0, L._capi.FOLD_BUF_T)
        # Montgomery -> canonical on the device (library kernel), then host
        t = wl.torch
        lib = L._capi.lib()
        both = t.from_numpy(np.concatenate([W2, T])).cuda()
        L._capi.check(lib.lurk_convert_dev(0, both.data_ptr(), both.numel() // 32, L.FMT_CANONICAL, both.data_ptr(), None))
        t.cuda.synchronize()
        both = both.cpu().numpy()
        W2c, Tc = both[:wl.nW * 32], both[wl.nW * 32:]
        if wl.key == "from_label":
            # the checker gets the key as data (a copy generated through the host-buffer entry point); 8 of its points are compared
            # with the Python restatement of from_label
            from oracle import h2c
            import hashlib
            nk = max(wl.nW, wl.nT)
            bases = L.from_label(CURVE, b"ck", nk)
            stream_ = hashlib.shake_256(b"ck").digest(32 * nk)
            for i in (0, 1, 65535, 65536, nk // 2, nk - 2, nk - 1, 12345):
                x = int.from_bytes(bases[64 * i:64 * i + 32].tobytes(), "little")
                y = int.from_bytes(bases[64 * i + 32:64 * i + 64].tobytes(), "little")
                assert (x, y) == h2c.hash_to_curve(CURVE, "from_uniform_bytes", stream_[32 * i:32 * i + 32]), i
            out["key_points_checked_against_oracle"] = 8
        else:
            bases = oracle.gen_bases(CURVE, max(wl.nW, wl.nT))
        want_w = oracle.msm(CURVE, bases, W2c, nthreads=th)
        want_t = oracle.msm(CURVE, bases, Tc, nthreads=th)
        r, h = spec.ro_squeeze(1, spec.nifs_absorb_list(PP_DIGEST, nifs.point_of(want_w), wl.X2, nifs.point_of(want_t)))
        nz_t = int(np.count_nonzero(Tc.reshape(-1, 32).any(axis=1)))
        out["oracle_fold"] = {"comm_W": bool(np.array_equal(rec.comm_W, want_w)), "comm_T": bool(np.array_equal(rec.comm_T, want_t)),
                              "challenge": int.from_bytes(rec.r.tobytes(), "little") == r, "terms": [wl.nW, wl.nT],
                              "cross_term_nonzero_fraction": round(nz_t / max(1, wl.nT), 4)}
    return out


def dump_outputs(wl, out_dir, sample=1 << 16):
    """writes what the last fold step handed its caller, per circuit: the step's record (fresh and running commitments,
    challenge, RO hash) and the running instance (W, E, u, X) it folded into, canonical form.  Every 32-byte field element
    becomes a row of eight little-endian 32-bit limbs stored as float64, which is exact.  W and E longer than `sample`
    elements keep a fixed seeded sample of their rows, so the whole dump stays a few MB."""
    os.makedirs(out_dir, exist_ok=True)
    limbs = lambda b: np.ascontiguousarray(b, dtype=np.uint8).view("<u4").reshape(-1, 8).astype(np.float64)
    for name, inst, rec in zip(wl.names, wl.inst, wl.last):
        arrays = {k: limbs(getattr(rec, k)) for k in ("comm_W", "comm_T", "r", "running_comm_W", "running_comm_E", "ro_hash")}
        run = inst.ctx.get_running()
        arrays["running_u"], arrays["running_X"] = limbs(run["u"]), limbs(run["X"])
        for k in ("W", "E"):
            v = limbs(run[k])
            if len(v) > sample:
                v = v[np.sort(np.random.default_rng(0).choice(len(v), sample, replace=False))]
            arrays["running_" + k] = v
        for k, v in arrays.items():
            np.save(os.path.join(out_dir, f"{name}_{k}.npy"), v)


def ncu_traffic():
    """dram bytes per launch of the dominant kernel from this round's committed ncu --set full capture (profiles/), or None"""
    import csv
    path = os.path.join(ROOT, "profiles", "r2_ncu_full_msm_accumulate_iso_raw.csv")
    try:
        rows = list(csv.reader(open(path)))
        hdr = rows[0]
        units = rows[1]
        best = None
        for row in rows[2:]:
            rec = dict(zip(hdr, row))
            if "msm_accumulate_kernel" not in rec.get("Kernel Name", ""):
                continue
            tot = 0.0
            for key in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                v = float(rec[key].replace(",", ""))
                u = units[hdr.index(key)].lower()
                tot += v * {"byte": 1, "kbyte": 1e3, "mbyte": 1e6, "gbyte": 1e9}.get(u, 1)
            best = tot
        return best
    except Exception:
        return None


def run_gpu(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        # NCCL may print a banner to stdout on the first communicator; stdout carries exactly one JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            warm = torch.zeros(1, device="cuda")
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    wl = FoldStepGPU(rank, world, scaling=args.scaling, latency_sms=args.latency_sms, workload=args.workload, rc=args.rc, key=args.key)
    wl.ctx.connect()          # exchange-buffer handles through the process group (setup only; the steps never call NCCL)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(staged, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            wl.step(staged)
        wl.drain()
        torch.cuda.synchronize()          # work runs on several streams: close the region after all of them drained
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    wl.start(staged=True)
    for _ in range(max(args.warmup, 3)):
        wl.step(True)
    wl.drain()
    verified = verify_full_size(wl, rank)          # after real folds, before timing
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms = timed(False, args.steps)
    stats = [i.ctx.stats() for i in wl.inst]
    st = stats[0]
    ms_e2e = timed(True, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(wl, args.dump_outputs)
    # the dominant kernel with nothing else on the GPU (inside the step it overlaps other streams' kernels)
    iso = []
    wl.ck_t.set_profiling(True)
    tbuf, tn = wl.ctx.device_buffer(0, wl.L._capi.FOLD_BUF_E1)     # the running error vector: full-width scalars on the rows T touches
    e_view = wl.ctx.device_view(0, wl.L._capi.FOLD_BUF_E1)[:wl.nT * 32].view(wl.nT, 32)
    iso_nonzero = int((e_view != 0).any(dim=1).sum().item())       # zero scalars never enter the bucket sort
    for _ in range(5):
        wl.ck_t.launch_device(tbuf, wl.nT, fmt=wl.L.FMT_MONTGOMERY, stream=0)
        wl.ck_t.finish()
        iso.append(wl.ck_t.last_profile()[0])
    iso = iso[2:]

    frames_total = wl.rc * world if args.scaling == "weak" else wl.rc
    iters = frames_total * args.steps
    value = iters / (ms / 1e3)
    e2e = iters / (ms_e2e / 1e3)
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        iso_ms = sum(iso) / max(1, len(iso))
        terms = wl.nT
        # algorithmic bytes of THIS launch: 96 B per non-zero term (scalar + base), 32 B per zero scalar (read and dropped)
        iso_bytes = iso_nonzero * 96 + (terms - iso_nonzero) * 32
        achieved = iso_bytes / (iso_ms / 1e3) / 1e9 if iso_ms > 0 else 0.0
        launches = sum(x["launches_a"] + x["launches_b"] for x in stats)
        out = {
            "metric": METRIC, "value": round(value, 2), "unit": "iterations/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(ms / args.steps, 4),
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "u32x8 (254-bit Montgomery integers)",
            "data": "synthetic", "config": workload_config(world, args.scaling, args.workload, wl.rc),
            "e2e": {"value": round(e2e, 2), "unit": "iterations/s", "h2d_bytes_per_step": int(wl.h2d_bytes),
                    "d2h_bytes_per_step": int(wl.d2h_bytes), "ms_per_step": round(ms_e2e / args.steps, 4)},
            "gpu_launches": int(launches * args.steps),
            "verified": verified,
            "roofline": {"kernel": "msm_accumulate_kernel (bucket accumulation of commit(T) / commit(W))", "bound": "hbm",
                         "achieved": round(achieved, 2), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 5),
                         "traffic": ncu_traffic(),
                         "traffic_note": "dram__bytes_read.sum + dram__bytes_write.sum of one launch in profiles/r2_ncu_full_msm_accumulate_iso_raw.csv (ncu --set full of "
                                         "this kernel on a DENSE 1114100-term vector and the c = 20 table, tools/acc_iso.py: 2.35 ms, 45.5 GB/s algorithmic); the launch "
                                         "timed here runs on the running error vector (terms_nonzero of terms) with commit(T)'s c = 16 table; Pippenger gathers each "
                                         "64-byte window multiple once per window",
                         "avg_launch_ms": round(iso_ms, 4), "avg_launch_ms_overlapped_in_step": {"commit_W": round(st["accumulate_w_ms"], 4),
                                                                                                "commit_T": round(st["accumulate_t_ms"], 4)},
                         "algorithmic_bytes_per_launch": int(iso_bytes), "terms": int(terms), "terms_nonzero": iso_nonzero,
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s",
                         "note": "bound by the FMA-heavy (IMAD.WIDE) pipe (ncu captures in profiles/): ~13 bucket additions x ~1.4e3 IMAD.WIDE "
                                 "per 96 algorithmic bytes; launch time = CUDA events inside the library on the launching stream, kernel run "
                                 "alone right after the timed region"},
            "clocks": clocks,
        }
        if args.key != "synthetic":
            out["config"]["key"] = "DlogGroup::from_label(b'ck') (hash-to-curve, generated on the GPU)"
            out["setup"] = {"ck_generate_ms": round(wl.ck_generate_ms, 1), "note": "outside the timed region (the metric excludes public-parameter setup)"}
        if args.latency_sms:
            out["config"]["sm_partition"] = f"{args.latency_sms} SMs reserved for the latency-shaped kernels (green contexts)"
        if world == 1 and not args.no_cpu_baseline and args.workload == "fib":
            out["cpu_baseline"] = cpu_baseline(sample_steps=1)
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------- CPU arm (oracle)
class FoldStepCPU:
    """the same fold on the host cores through the oracle (plain C + OpenMP for the vectors, Python for the few scalars)"""

    def __init__(self, frames, threads, seed=0x6c75726b):
        from oracle import capi as oracle, nifs
        self.o, self.nifs, self.th, self.frames = oracle, nifs, threads, frames
        rng = np.random.default_rng(seed)
        mats, self.nW, self.nT, prod_rows = step_circuit(seed, frames)
        self.bases = oracle.gen_bases(CURVE, max(self.nW, self.nT))
        self.prim = nifs.NovaOracle(CURVE, self.bases, mats, self.nW, 2, nthreads=threads, pp_digest=PP_DIGEST)
        mats2, self.nW2, self.nT2, _ = step_circuit(seed + 7, 1, slot_elems=SECONDARY_N - 1500, glue=1500, cons=SECONDARY_N)
        self.sec = nifs.NovaOracle(CURVE2, oracle.gen_bases(CURVE2, max(self.nW2, self.nT2)), mats2, self.nW2, 2, nthreads=threads, pp_digest=PP_DIGEST)
        self.slot_pre = {}
        for arity, per_frame in SLOTS:
            n = frames * per_frame
            pre = rand_elements(rng, n * arity).reshape(n, arity * 32)
            pre[rng.random(n) >= LIVE_SLOT_FRACTION] = 0
            self.slot_pre[arity] = pre.reshape(-1)
            oracle.install_params(0, arity)
        self.bd = rand_elements(rng, frames * BITDECOMP_PER_FRAME, "witness")
        self.offs = None
        self.W2 = rand_elements(rng, self.nW, "witness")
        self.W2s = rand_elements(rng, self.nW2, "witness")
        self.X2 = [3, 5]
        self.prim.init_running(self.W2, self.X2)
        self.sec.init_running(self.W2s, self.X2)

    def step(self):
        o, th = self.o, self.th
        parts = [o.poseidon_witness_batch(0, a, self.slot_pre[a], nthreads=th) for a, _ in SLOTS]
        parts.append(o.bitdecomp_witness_batch(0, self.bd, nthreads=th))
        slots = np.concatenate(parts)
        self.W2[:slots.size] = slots             # same element count as the frame layout; positions do not change the work
        self.prim.prove_step(self.W2, self.X2)
        self.sec.prove_step(self.W2s, self.X2)


def host_threads():
    """all the host threads the box has -- NOT omp_get_max_threads(): torchrun exports OMP_NUM_THREADS=1"""
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_baseline(sample_steps=1, frames=RC):
    """bounded sample of the same workload on the host cores (oracle = CPU port of the reference path)"""
    th = host_threads()
    wl = FoldStepCPU(frames, th)
    t0 = time.perf_counter()
    for _ in range(sample_steps):
        wl.step()
    dt = time.perf_counter() - t0
    return {"value": round(frames * sample_steps / dt, 3), "unit": "iterations/s", "cores": th, "kind": "port",
            "sample": f"{sample_steps} fold step(s) of {frames} frames ({dt:.1f} s): oracle/oracle.c (4x64-bit Montgomery + OpenMP) + oracle/nifs.py; "
                      "the reference's Rust prover (hand-written asm MSM) cannot be built in this image"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    th = host_threads()
    wl = FoldStepCPU(RC, th)
    # with SMT the oracle is sometimes faster on one thread per core -- time one warm-up step each way and keep the faster
    best = None
    for t in sorted({th, max(1, th // 2)}, reverse=True):
        wl.th = wl.prim.th = wl.sec.th = t
        t0 = time.perf_counter()
        wl.step()
        dt1 = time.perf_counter() - t0
        if best is None or dt1 < best[0]:
            best = (dt1, t)
    wl.th = wl.prim.th = wl.sec.th = best[1]
    steps = args.steps          # each step is ~2 s on 64 cores, ~8 s on 8
    for _ in range(max(0, min(args.warmup, 3) - 2)):
        wl.step()
    t0 = time.perf_counter()
    for _ in range(steps):
        wl.step()
    dt = time.perf_counter() - t0
    value = RC * steps / dt
    sample = (f"{steps} timed fold step(s) of {RC} frames each (one rank's share of the workload; per-frame cost does not depend on the frame count), "
              f"{wl.th} host threads, oracle/oracle.c + oracle/nifs.py (CPU port; upstream Rust prover not buildable here)")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": round(value, 3),
        "unit": "iterations/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(dt / steps * 1e3, 2), "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "u64x4 (254-bit Montgomery integers)", "data": "synthetic", "config": workload_config(world, args.scaling),
        "cpu_baseline": {"value": round(value, 3), "unit": "iterations/s", "cores": wl.th, "kind": "port", "sample": sample},
        "e2e": {"value": round(value, 3), "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def main():
    global LIVE_SLOT_FRACTION
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N > 1: weak = rc 100 per GPU (rc = 100 N step circuit); strong = ONE rc = 100 fold, its key split N ways")
    ap.add_argument("--latency-sms", type=int, default=0, help="SM partition (green contexts): SMs reserved for the chain's latency-shaped kernels")
    ap.add_argument("--workload", default="fib", choices=["fib", "sha256_ivc", "trie_nivc"],
                    help="fib = the BASELINE metric (benches/fibonacci.rs rc=100); sha256_ivc / trie_nivc = BASELINE configs[3] / configs[4] shapes")
    ap.add_argument("--rc", type=int, default=None, help="frames per step (default: 100 fib, 10 sha256_ivc, 400 trie_nivc)")
    ap.add_argument("--live-slots", type=float, default=LIVE_SLOT_FRACTION,
                    help="fraction of a frame's slots with a non-dummy preimage (dummy slots share one witness, multiframe.rs:553-577)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--key", default="synthetic", choices=["synthetic", "from_label"],
                    help="commitment key: [i+1]G (default; the CPU arm uses the same) or the reference's hash-to-curve key generated on the GPU (N3)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last fold step's outputs as DIR/<name>.npy (float64; GPU arm only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm (--impl b200)")
    LIVE_SLOT_FRACTION = args.live_slots
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
