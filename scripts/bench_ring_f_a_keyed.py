"""Ring f_a with a key per target (qf_ring_set_key_table + qf_ring_f_a_keyed_dev, DESIGN.md 4.13) at C3 (X^256 + 1,
q = 3329, k = 12: 14 polynomials, D = 3584).

sigma comes from qf_samp_d_dev and stays on the device (262 144 targets per pass, 3.8 GB: far larger than the 126 MB L2).
Measured, each variant alternating with the others in each of two rounds (CUDA events; 2 warm-up passes, then enough timed
passes for about half a second):
  - keyed evals/s for T = 1, 236, 4096 and 65 536 uniform keys, key indices in random order and sorted by key;
  - unkeyed qf_f_a_dev on the dense tensor-core path and on the ring_small NTT path (QF_DISABLE_RING_DENSE=1);
  - qf_ring_set_key_table for 4096 and 65 536 keys against qf_ring_set_a per key (a loop over 128 keys, per-key time);
  - qf_ring_trap_gen_batch_from for 4096 keys against qf_ring_trap_gen_from per key (a loop over 128 keys).
Every timed keyed output is checked: a seeded sample of 32 rows against f_a with the row's own key installed.  Writes one
JSON file with the card name and power limit.

  python scripts/bench_ring_f_a_keyed.py [--out FILE] [--quick]
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N, Q = 256, 3329
KEY_COUNTS = (1, 236, 4096, 65536)
SAMPLE = 32


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in out.split(",")]
    return {"name": name, "power_limit": power}


def timed(torch, fn, min_s):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    one = a.elapsed_time(b) / 1e3
    reps = max(1, min(1000, int(math.ceil(min_s / max(one, 1e-6)))))
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / 1e3 / reps


T0 = time.perf_counter()


def log(msg):
    print(f"[{time.perf_counter() - T0:7.1f} s] {msg}", flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_ring_f_a_keyed.json"))
    ap.add_argument("--quick", action="store_true", help="small batch and short windows (rehearsal)")
    args = ap.parse_args()

    import torch

    import tools_b200 as T
    from tools_b200 import _ffi

    B = 16384 if args.quick else 262144
    min_s = 0.1 if args.quick else 0.5
    rounds = 1 if args.quick else 2
    gp = T.GadgetParametersRing.init_default(N, Q)
    s = ((2 * 2 * 1.005 * math.sqrt(N) + 1) * 2) * 4
    d = N * (gp.k + 2)
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(1)
    res = {"gpu": gpu_info(), "workload": f"C3 ring f_a, n = {N}, q = {Q}, k = {gp.k}, D = {d}, {B} targets per pass, "
                                          "sigma device-resident (qf_samp_d_dev)", "batch": B}

    psf = T.PSFGPVRing(gp, s, 1.005)
    check = T.PSFGPVRing(gp, s, 1.005)  # plain f_a with one key installed (dense path): the reference of the checks
    os.environ["QF_DISABLE_RING_DENSE"] = "1"
    small = T.PSFGPVRing(gp, s, 1.005)  # its qf_ring_set_a reads the switch: the ring_small path for unkeyed f_a
    small._install_a(rng.integers(0, Q, (gp.k + 2, N), dtype=np.int64))
    del os.environ["QF_DISABLE_RING_DENSE"]

    stream = torch.cuda.current_stream(dev).cuda_stream  # the library runs where the CUDA events are recorded
    for p in (psf, small, check):
        p.ctx.call("qf_set_stream", _ffi.ptr(stream))
    sig = torch.empty((B, d), dtype=torch.int32, device=dev)
    u = torch.empty((B, N), dtype=torch.int64, device=dev)
    fl = torch.empty(B, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    psf.ctx.call("qf_samp_d_dev", B, 5, 0, _ffi.ptr(sig.data_ptr()))
    psf.ctx.call("qf_synchronize")
    sample = rng.choice(B, SAMPLE, replace=False)
    log("sigma ready")

    # key tables (installed once per T; installs timed below)
    tables = {}
    for t in KEY_COUNTS:
        keys = rng.integers(0, Q, (t, gp.k + 2, N), dtype=np.int64)
        idx = rng.integers(0, t, B).astype(np.int32)
        order = np.argsort(idx, kind="stable")
        tables[t] = dict(keys=keys, idx=torch.from_numpy(idx).to(dev), idx_sorted=torch.from_numpy(idx[order]).to(dev),
                         sig_sorted=None, order=order)
    a0 = rng.integers(0, Q, (gp.k + 2, N), dtype=np.int64)
    psf._install_a(a0)
    log("keys and indices ready")

    def keyed(ctx, sg, ix):
        return lambda: ctx.call("qf_ring_f_a_keyed_dev", _ffi.ptr(sg.data_ptr()), _ffi.ptr(ix.data_ptr()), B,
                                _ffi.ptr(u.data_ptr()), _ffi.ptr(fl.data_ptr()))

    def unkeyed(p):
        return lambda: p.ctx.call("qf_f_a_dev", _ffi.ptr(sig.data_ptr()), B, _ffi.ptr(u.data_ptr()), _ffi.ptr(fl.data_ptr()))

    def verify(keys, sg, ix):
        psf.ctx.call("qf_synchronize")
        assert bool(fl.all())
        uh, ih = u[sample].cpu().numpy(), ix[sample].cpu().numpy()
        sh = sg[sample].cpu().numpy().reshape(SAMPLE, gp.k + 2, N)
        for j in range(SAMPLE):
            want, _ = check.f_a_batch(keys[ih[j]], sh[j:j + 1])
            assert np.array_equal(want[0], uh[j]), "keyed f_a differs from f_a with the row's own key"

    rates = {}
    for rd in range(rounds):
        for name, p in (("unkeyed_dense", psf), ("unkeyed_ring_small", small)):
            dt = timed(torch, unkeyed(p), min_s)
            rates.setdefault(name, []).append(B / dt)
            log(f"round {rd} {name}: {B / dt / 1e6:.1f} M evals/s")
        for t in KEY_COUNTS:
            tb = tables[t]
            psf.ctx.call("qf_ring_set_key_table", _ffi.ptr(np.ascontiguousarray(tb["keys"])), t)
            if tb["sig_sorted"] is None:
                tb["sig_sorted"] = sig[torch.from_numpy(tb["order"]).to(dev)].contiguous()
            for mode, sg, ix in (("random", sig, tb["idx"]), ("sorted", tb["sig_sorted"], tb["idx_sorted"])):
                dt = timed(torch, keyed(psf.ctx, sg, ix), min_s)
                verify(tb["keys"], sg, ix)
                rates.setdefault(f"keyed_T{t}_{mode}", []).append(B / dt)
                log(f"round {rd} keyed T = {t} {mode}: {B / dt / 1e6:.1f} M evals/s")
            tb["sig_sorted"] = None  # one extra copy of sigma at a time
            torch.cuda.empty_cache()
    res["evals_per_s"] = {k: {"rounds": v, "mean": float(np.mean(v))} for k, v in rates.items()}

    log("installs")
    inst = {}
    for t in (4096, 65536):
        keys = np.ascontiguousarray(tables[t]["keys"])
        ts = []
        for _ in range(2):
            t0 = time.perf_counter()
            psf.ctx.call("qf_ring_set_key_table", _ffi.ptr(keys), t)
            ts.append(time.perf_counter() - t0)
        inst[f"set_key_table_{t}_s"] = min(ts)
    loop = 16 if args.quick else 128
    keys = tables[4096]["keys"]
    t0 = time.perf_counter()
    for j in range(loop):
        psf.ctx.call("qf_ring_set_a", _ffi.ptr(np.ascontiguousarray(keys[j])))
    per = (time.perf_counter() - t0) / loop
    inst["ring_set_a_per_key_s"] = per
    inst["ring_set_a_loop_projected_4096_s"] = per * 4096
    inst["ring_set_a_loop_projected_65536_s"] = per * 65536
    res["install"] = inst

    log(f"installs: {inst}")
    cnt = 4096
    a_bars = rng.integers(0, Q, (cnt, N), dtype=np.int64)
    rs = rng.integers(-4, 5, (cnt, gp.k, N)).astype(np.int32)
    es = rng.integers(-4, 5, (cnt, gp.k, N)).astype(np.int32)
    ts = []
    for _ in range(2):
        t0 = time.perf_counter()
        got = psf.gen_trapdoor_ring_lwe_batch(a_bars, rs, es)
        ts.append(time.perf_counter() - t0)
    t0 = time.perf_counter()
    for j in range(loop):
        one = check.gen_trapdoor_ring_lwe(a_bars[j], rs[j], es[j])
        assert np.array_equal(one, got[j])
    per = (time.perf_counter() - t0) / loop
    res["trap_gen"] = {"batch_4096_s": min(ts), "single_per_key_s": per, "single_loop_projected_4096_s": per * 4096}
    log(f"trap_gen: {res['trap_gen']}")

    res["note"] = ("evals/s = targets / (time of one qf_*_dev call over the batch, CUDA events); 'sorted' permutes sigma "
                   "and the indices by key beforehand (not timed).  Install and TrapGen times are host wall clock of the "
                   "synchronous calls; the qf_ring_set_a and qf_ring_trap_gen_from loops ran over " + str(loop) +
                   " keys and are projected linearly.")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1), flush=True)


if __name__ == "__main__":
    main()
