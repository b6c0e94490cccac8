#!/usr/bin/env python3
"""GPU time of `compress` with one reduced polynomial opening against one opening per evaluation claim.

--workload trie_nivc: SuperNova (reference src/proof/supernova.rs:110,293-317 -> BatchedRelaxedR1CSSNARK): the Lurk step circuit of
bench.py at --rc frames (LURK_FRAME, 400 by default) plus the trie-lookup coprocessor circuit (TRIE_LOOKUP), proven by
BatchedRelaxedR1CSProver.  --workload fib: Nova (src/proof/nova.rs:92 -> RelaxedR1CSSNARK), one Lurk step circuit at --rc frames
(100 by default), proven by RelaxedR1CSProver.  Random z / E as in tools/compress_bench.py: the prover's cost does not depend on
satisfiability (tests/test_gpu_spartan_batched.py checks real folded instances against the verifiers at small sizes).

In the same process, alternating rep by rep, it times
  (a) the chain ending in batch_eval_prove: the 2k evaluation claims reduced to one joint polynomial, ONE HyperKZG opening;
  (b) the same chain ending in one HyperKZG opening per claim (2k openings), as the chain did before the reduction existed.
Both under a powers-of-tau key of 2^m_max points with its fixed-base table.  One JSON object per line: the card's name and power
limit, then per variant and phase the median / min wall-clock (device synchronise at each phase end) over --reps reps, then the
totals.  The transcript is a Python stand-in (sha256), so every sum-check round includes a Python callback."""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (the step-circuit generator and circuit shapes)
import lurk_beta_b200 as L  # noqa: E402

CURVE, FIELD = 0, 0


def challenge(label, data):
    return int.from_bytes(hashlib.sha256(repr((label, data)).encode()).digest()[:30], "little")


def rand_mont(n, seed):
    rng = np.random.default_rng(seed)
    raw = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    raw[:, 31] &= 0x1f
    return torch.from_numpy(raw.reshape(-1)).cuda()


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in out.split(",")]
    except Exception as e:                   # the numbers stay valid; the card's settings are then unknown
        info["power_limit"] = f"unknown ({type(e).__name__})"
    return info


def circuits(workload, rc):
    """[(name, mats, n_w)]: bench.py's synthetic step circuits"""
    shape = bench.LURK_FRAME
    mats, n_w, _, _ = bench.step_circuit(1, rc, slot_elems=bench.SLOT_ELEMS, glue=shape["glue"], cons=shape["cons"])
    out = [("lurk step", mats, n_w)]
    if workload == "trie_nivc":
        t = bench.TRIE_LOOKUP
        _, t_slots = bench.slot_offsets(1, 0, t["slots"], t["bd"], FIELD)
        mats, n_w, _, _ = bench.step_circuit(2, 1, slot_elems=t_slots, glue=t["glue"], cons=t["cons"])
        out.append(("trie lookup", mats, n_w))
    return out


def hyperkzg(ck):
    return lambda d_P, point, value: L.spartan.hyperkzg_prove(CURVE, ck, d_P.data_ptr(), point, lambda r, m: challenge("pcs", (r, bytes(m[:64]))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="trie_nivc", choices=["trie_nivc", "fib"])
    ap.add_argument("--rc", type=int, default=None, help="frames of the Lurk step circuit (default: 400 trie_nivc, 100 fib)")
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    rc = a.rc or {"trie_nivc": 400, "fib": 100}[a.workload]
    print(json.dumps(dict(gpu_info(), workload=a.workload, rc=rc)), flush=True)
    t0 = time.perf_counter()
    provers, shapes = [], []
    for name, mats, n_w in circuits(a.workload, rc):
        pr = L.spartan.RelaxedR1CSProver(FIELD, mats, n_w, 2)
        provers.append(pr)
        shapes.append(dict(circuit=name, constraints=pr.rows, variables=n_w, rows_padded_log2=pr.log_rows, vars_padded_log2=pr.num_vars.bit_length() - 1,
                           nnz=[int(m[0][-1]) for m in mats]))
    inputs = []
    for i, pr in enumerate(provers):
        z = pr.pad_z(rand_mont(pr.n_w, 10 * i + 1), 12345 + i, [6, 7])
        inputs.append((z, rand_mont(pr.rows, 10 * i + 2), 12345 + i, [6, 7]))
    m_max = max(max(pr.log_rows, pr.num_vars.bit_length() - 1) for pr in provers)
    torch.cuda.synchronize()
    setup_s = time.perf_counter() - t0
    g = L.synthetic_bases(0, 1, start=9)
    gi = (int.from_bytes(g[:32].tobytes(), "little"), int.from_bytes(g[32:].tobytes(), "little"))
    t0 = time.perf_counter()
    ck = L.CommitmentKey.powers_of_tau(CURVE, gi, 987654321987654321, 1 << m_max)
    ck.precompute()
    torch.cuda.synchronize()
    key_ms = (time.perf_counter() - t0) * 1e3
    print(json.dumps(dict(workload=a.workload, circuits=shapes, claims=2 * len(provers), key_points_log2=m_max,
                          setup={"matrices_to_device_and_transposes_s": round(setup_s, 2), "key_and_fixed_base_table_ms": round(key_ms, 1)})), flush=True)
    batched = L.spartan.BatchedRelaxedR1CSProver(provers) if a.workload == "trie_nivc" else None

    def chain(timings):
        """the Spartan chain up to the 2k evaluation claims"""
        if batched is not None:
            return batched.prove(inputs, challenge, timings=timings)["eval_claims"]
        pr, (z, dE, u, _) = provers[0], inputs[0]
        proof = pr.prove(z, dE, u, challenge, timings)
        return [(z, proof["ry"][1:], proof["eval_W"]), (proof["E_padded"], proof["rx"], proof["claims"][3])]

    def reduced():
        timings = {}
        t0 = time.perf_counter()
        claims = chain(timings)
        t1 = time.perf_counter()
        L.spartan.batch_eval_prove(FIELD, claims, challenge, hyperkzg(ck))
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        timings[f"batch_eval_reduce + 1 opening (2^{m_max})"] = (t2 - t1) * 1e3
        return (t2 - t0) * 1e3, timings

    def per_claim():
        timings = {}
        t0 = time.perf_counter()
        claims = chain(timings)
        t1 = time.perf_counter()
        for d_P, point, _ in claims:
            hyperkzg(ck)(d_P, point, None)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        timings[f"{len(claims)} openings (" + ", ".join(f"2^{len(pt)}" for _, pt, _ in claims) + ")"] = (t2 - t1) * 1e3
        return (t2 - t0) * 1e3, timings

    variants = {"one reduced opening": reduced, "one opening per claim": per_claim}
    for fn in variants.values():           # warm-up: module loads, scratch pools, every shape of the timed window
        fn()
    runs = {name: [] for name in variants}
    for _ in range(a.reps):
        for name, fn in variants.items():
            runs[name].append(fn())
    for name, rs in runs.items():
        for phase in rs[0][1]:
            xs = [r[1][phase] for r in rs]
            print(json.dumps(dict(workload=a.workload, rc=rc, variant=name, phase=phase, median_ms=round(statistics.median(xs), 3),
                                  min_ms=round(min(xs), 3), reps=len(xs))), flush=True)
    totals = {name: statistics.median(r[0] for r in rs) for name, rs in runs.items()}
    print(json.dumps(dict(workload=a.workload, rc=rc, total_median_ms={k: round(v, 2) for k, v in totals.items()},
                          saved_ms=round(totals["one opening per claim"] - totals["one reduced opening"], 2), reps=a.reps,
                          note="wall-clock, device synchronise at each phase end; variants alternate rep by rep; Python stand-in transcript")),
          flush=True)


if __name__ == "__main__":
    main()
