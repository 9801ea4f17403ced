"""Offline / online samp_p (qf_samp_p_offline + qf_samp_p_online_dev; DESIGN.md 4.12) against qf_samp_p_dev.

Two workloads, device-resident targets:
  c2  PSFGPV n = 256, q = 2^24, m = 12352 on the two-phase recursion, one bench.py step of 227 328 targets
  c4  one C4 shard: PSFPerturbation n = 512, q = 2^32 - 5, m = 32849, r = 9, structured sqrt(Sigma_2), 60 416 targets
Measured per workload (host clock around work that ends in a device synchronise; the variants alternate within each
round and every shape is run once before the timed rounds):
  step     qf_samp_p_dev on the full step against qf_samp_p_offline + qf_samp_p_online_dev for the same count: the total
           cost of the split and the online share
  latency  online_dev against samp_p_dev for batches of 1, 128, 1024 and 8192 targets (the pool filled beforehand, outside
           the timed window), untagged and with one polynomial tag per target (qf_samp_p_tagged_dev)
Every timed output is checked: A e = u (A_t e = u, by qf_f_a_tagged_dev with a polynomial f_a table of the same tags)
exactly on every row, on the device.  Prints one JSON line with the card name and power limit read in the same run.

  python scripts/bench_offline_online.py [--workloads c2,c4] [--rounds 3] [--out FILE]
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

BATCHES = (1, 128, 1024, 8192)


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in out.split(",")]
    return {"name": name, "power_limit": power}


def setup(T, name):
    if name == "c4":
        n, q, r = 512, 2**32 - 5, 9.0
        gp = T.GadgetParameters.init_default(n, q)
        s1 = (math.sqrt(gp.m_bar) + math.sqrt(n * gp.k)) / math.sqrt(2)
        psf = T.PSFPerturbation(gp, r, float(math.ceil(1.15 * math.sqrt(5 * (s1 * s1 + 1) + 1))))
        a, td = psf.trap_gen(seed=2, dense_sqrt_sigma_2=False)
        B = 60416
    else:
        n, q = 256, 2**24
        gp = T.GadgetParameters.init_default(n, q)
        psf = T.PSFGPV(gp, float(math.ceil((math.sqrt(gp.m_bar) + 1.0) * math.sqrt(5.0) * math.log2(n))))
        a, td = psf.trap_gen(seed=2, dense_gso=False)
        B = 227328
    psf._install_a(a)
    psf._install_td(a, td)
    return gp, psf, a, td, B


def poly_tags(T, rng, count, n, q):
    h = rng.integers(0, q, (count, n), dtype=np.int64)
    if q % 2 == 0:  # X^n + 1 = (X + 1)^n mod 2: h is a unit iff h(1) is odd
        h[:, 0] += (h.sum(axis=1) + 1) % 2
        h %= q
    f = np.zeros(n, dtype=np.int64)
    f[0] = 1
    return T.PolyTags(f, h)


def run_workload(T, name, args):
    import torch

    from tools_b200 import _ffi

    gp, psf, a, td, B = setup(T, name)
    n, m, q = gp.n, gp.m, gp.q
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(7)
    u = torch.from_numpy(rng.integers(0, q, (B, n), dtype=np.int64)).to(dev)
    e = torch.empty((B, m), dtype=torch.int32, device=dev)
    uo = torch.empty((B, n), dtype=torch.int64, device=dev)
    flags = torch.empty(B, dtype=torch.uint8, device=dev)
    Tn = max(BATCHES)
    tags = poly_tags(T, rng, Tn, n, q)
    psf.set_tag_table(a, td, tags)
    psf._install_fa_tags(tags, None)
    tidx = torch.arange(Tn, dtype=torch.int32, device=dev)
    ptr = lambda t: _ffi.ptr(t.data_ptr())  # noqa: E731
    seed, index = 11, [0]
    checks = {"rows_checked": 0, "all_exact": True}

    def check(rows, tagged):
        """A e = u (A_t e = u) on every row of the last output, on the device."""
        if tagged:
            psf.ctx.call("qf_f_a_tagged_dev", ptr(e), ptr(tidx), rows, ptr(uo), ptr(flags))
        else:
            psf.ctx.call("qf_f_a_dev", ptr(e), rows, ptr(uo), ptr(flags))
        psf.ctx.call("qf_synchronize")
        ok = bool(torch.equal(uo[:rows], u[:rows])) and bool(flags[:rows].all())
        checks["rows_checked"] += rows
        checks["all_exact"] = checks["all_exact"] and ok
        assert ok, (name, rows, tagged)

    def direct(rows, tagged):
        index[0] += rows
        t0 = time.perf_counter()
        if tagged:
            psf.ctx.call("qf_samp_p_tagged_dev", ptr(u), ptr(tidx), rows, seed, index[0], ptr(e))
        else:
            psf.ctx.call("qf_samp_p_dev", ptr(u), rows, seed, index[0], ptr(e))
        psf.ctx.call("qf_synchronize")
        dt = time.perf_counter() - t0
        check(rows, tagged)
        return dt

    def fill(rows):
        index[0] += rows
        t0 = time.perf_counter()
        psf.ctx.call("qf_samp_p_offline", rows, seed, index[0])
        return time.perf_counter() - t0

    def online(rows, tagged):
        t0 = time.perf_counter()
        psf.ctx.call("qf_samp_p_online_dev", ptr(u), ptr(tidx) if tagged else None, rows, ptr(e), None)
        psf.ctx.call("qf_synchronize")
        dt = time.perf_counter() - t0
        check(rows, tagged)
        return dt

    res = {"targets_per_step": B, "step": {}, "latency": {}}
    # ---- full step: composed against fill + online
    direct(B, False)
    fill(B), online(B, False)  # warm-up of both shapes
    t_direct, t_fill, t_online = [], [], []
    for _ in range(args.rounds):
        t_direct.append(direct(B, False))
        t_fill.append(fill(B))
        t_online.append(online(B, False))
    md, mf, mo = (float(np.median(x)) for x in (t_direct, t_fill, t_online))
    res["step"] = {"samp_p_dev_s": md, "offline_s": mf, "online_dev_s": mo, "split_total_over_direct": (mf + mo) / md,
                   "online_over_direct": mo / md, "online_share_of_split": mo / (mf + mo),
                   "samples": {"samp_p_dev": t_direct, "offline": t_fill, "online_dev": t_online}}
    # ---- latency: one pool for all batch sizes of a round, filled outside the timed windows
    for tagged in (False, True):
        for b in BATCHES:
            direct(b, tagged)
        fill(sum(BATCHES) * (args.rounds + 1))
        for b in BATCHES:
            online(b, tagged)
        rows = {b: {"samp_p_dev": [], "online_dev": []} for b in BATCHES}
        for _ in range(args.rounds):
            for b in BATCHES:
                rows[b]["samp_p_dev"].append(direct(b, tagged))
                rows[b]["online_dev"].append(online(b, tagged))
        key = "poly_tag_per_target" if tagged else "untagged"
        res["latency"][key] = {
            str(b): {"samp_p_dev_ms": 1e3 * float(np.median(r["samp_p_dev"])), "online_dev_ms": 1e3 * float(np.median(r["online_dev"])),
                     "online_over_direct": float(np.median(r["online_dev"]) / np.median(r["samp_p_dev"]))}
            for b, r in rows.items()}
    res["checks"] = checks
    psf.ctx.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c2,c4")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_offline_online.json"))
    args = ap.parse_args()
    import tools_b200 as T

    out = {"gpu": gpu_info(), "rounds": args.rounds, "timing": "host clock around work ending in a device synchronise; "
           "median over rounds; variants alternate within a round", "workloads": {}}
    for w in args.workloads.split(","):
        out["workloads"][w] = run_workload(T, w, args)
        print(f"[{w}] {json.dumps(out['workloads'][w]['step'])}", file=sys.stderr, flush=True)
    out["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
