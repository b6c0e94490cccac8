"""bench.py contract: the reference arm runs on CPU and prints exactly one JSON line with the required keys; the committed
record of the B200 arm carries the keys the driver and the judge read."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
             "dtype", "data", "config", "e2e"}


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert BASE_KEYS <= set(d) and d["impl"] == "reference"
    assert d["unit"] == "iterations/s" and d["higher_is_better"] is True and d["value"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and "sample" in cb and cb["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_committed_b200_record_has_contract_keys():
    d = json.load(open(os.path.join(ROOT, "profiles", "r1_bench_n1.json")))
    assert BASE_KEYS | {"gpu_launches", "roofline", "cpu_baseline", "clocks"} <= set(d)
    r = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and r["bound"] in ("hbm", "tensor")
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-4
    assert d["gpu_launches"] > 0 and d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    assert d["metric"].startswith("Lurk iterations proved/sec") and d["config"]["workload"]


def test_dump_outputs_writes_exact_float64_limbs(tmp_path):
    """--dump-outputs: every field element becomes eight exact 32-bit limbs in float64; long W / E keep a seeded sample of rows"""
    import numpy as np
    from types import SimpleNamespace
    sys.path.insert(0, ROOT)
    import bench
    rng = np.random.default_rng(3)
    elems = lambda n: rng.integers(0, 256, size=n * 32, dtype=np.uint8)
    rec = SimpleNamespace(comm_W=elems(3), comm_T=elems(3), r=elems(1), running_comm_W=elems(3), running_comm_E=elems(3), ro_hash=elems(1))
    run = dict(W=elems(100), E=elems(30), u=elems(1), X=elems(2))
    ctx = SimpleNamespace(get_running=lambda: run)
    wl = SimpleNamespace(names=["primary"], inst=[SimpleNamespace(ctx=ctx)], last=[rec])
    for out in (tmp_path / "a", tmp_path / "b"):
        bench.dump_outputs(wl, str(out), sample=40)
    to_bytes = lambda a: a.astype("<u4").tobytes()
    for k in ("comm_W", "comm_T", "r", "running_comm_W", "running_comm_E", "ro_hash"):
        a = np.load(tmp_path / "a" / f"primary_{k}.npy")
        assert a.dtype == np.float64 and a.shape[1] == 8 and to_bytes(a) == getattr(rec, k).tobytes()
    assert to_bytes(np.load(tmp_path / "a" / "primary_running_E.npy")) == run["E"].tobytes()
    assert to_bytes(np.load(tmp_path / "a" / "primary_running_X.npy")) == run["X"].tobytes()
    w = np.load(tmp_path / "a" / "primary_running_W.npy")
    assert w.shape == (40, 8) and np.array_equal(w, np.load(tmp_path / "b" / "primary_running_W.npy"))
    rows = {to_bytes(w[i:i + 1]) for i in range(40)}
    assert len(rows) == 40 and rows <= {run["W"][32 * i:32 * i + 32].tobytes() for i in range(100)}


def test_synthetic_step_circuit_is_satisfiable_by_construction():
    """bench.py's full-size R1CS generator (vectorised) obeys the rule it documents: with the glue columns defined by the
    product rows, any slot-column content satisfies (A z) o (B z) = (C z); checked on the oracle at a small size"""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    from oracle import capi, nifs, spec
    frames, slot_elems, glue, cons = 3, 40, 9, 31
    mats, n_w, rows, prod_rows = bench.step_circuit(5, frames, slot_elems=slot_elems, glue=glue, cons=cons)
    assert (n_w, rows, len(prod_rows)) == (frames * (slot_elems + glue), frames * cons, frames * glue)
    p = spec.FIELD_MODULUS[0]
    rng = np.random.default_rng(1)
    W = [int(rng.integers(0, 2**62)) * int(rng.integers(0, 2**62)) % p for _ in range(n_w)]
    per = slot_elems + glue
    for f in range(frames):
        for g in range(glue):
            W[f * per + slot_elems + g] = 0
    X = [11, 13]
    z = nifs.pack(W + [1] + X)
    az, bz = (nifs.ints(capi.spmv(0, rp, col, val, z)) for rp, col, val in mats[:2])
    for k, row in enumerate(prod_rows):                      # the LEM-body aux stand-in: glue_g = (A_g . z)(B_g . z)
        f, g = divmod(k, glue)
        assert row == f * cons + g
        W[f * per + slot_elems + g] = az[row] * bz[row] % p
    o = nifs.NovaOracle(0, capi.gen_bases(0, max(n_w, rows)), mats, n_w, 2)
    assert o.bad_rows(nifs.pack(W), np.zeros(rows * 32, dtype=np.uint8), 1, X) == 0
    c = int(mats[0][1][0])                                   # a slot column that the first defining row reads
    W[c] = (W[c] + 1) % p
    assert o.bad_rows(nifs.pack(W), np.zeros(rows * 32, dtype=np.uint8), 1, X) > 0
