"""PSFGPV samp_p with a tag per target (qf_set_tag_table + qf_samp_p_tagged_dev on the two-phase recursion, DESIGN.md 4.3)
against the plain identity key, and the PSFGPV tag switch (qf_gpv_set_tag) against re-installing the switched key.

C2 (PSFGPV n = 256, q = 2^24, m = 12352, s as in bench.py), device-resident, 227 328 targets per step, 3 warm-up and 4
timed steps per variant (CUDA events), the variants alternating in each of two rounds on one context:
  identity   qf_samp_p_dev on the identity key A = [A_bar | G - A_bar R]
  T=1        qf_samp_p_tagged_dev with a table of one tag
  T=236      236 tags (about 960 targets per tag)
  T=4096     4096 tags (about 55 targets per tag)
Tags are random upper unitriangular, tag indices shuffled.  On every timed output A_t e = u is checked exactly on a seeded
sample of 512 rows on the host (A_t e = A e + (H_t - I) G e_bot, bench_tag_table.Checker).  Also times, with a host clock
around synchronised calls: qf_set_tag_table for T = 236 and 4096; qf_gpv_set_tag without and with s_out (the new short
basis); and qf_set_a + qf_set_trapdoor_gpv of the switched key (what a caller does without the switch).  Prints one JSON
line, with the card name and power limit.

  python scripts/bench_gpv_tag_table.py [--out FILE]
  python scripts/bench_gpv_tag_table.py --kernel-time   # a run of its own: torch.profiler (CUDA activities) time of the
                                                        # per-target tag kernel per step
"""
import argparse
import json
import math
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from bench_tag_table import Checker, gpu_info, unitriangular_tags  # noqa: E402


def setup():
    import tools_b200 as T

    n, q = 256, 2**24
    gp = T.GadgetParameters.init_default(n, q)
    s = float(math.ceil((math.sqrt(gp.m_bar) + 1.0) * math.sqrt(5.0) * math.log2(n)))  # bench.py gpv_s
    psf = T.PSFGPV(gp, s)
    a, td = psf.trap_gen(seed=2, dense_gso=False)
    psf._install_a(a)
    psf._install_td(a, td)
    return T, gp, s, psf, a, td


def sync_time(f):
    t0 = time.time()
    f()
    return time.time() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=227328)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--tables", default="1,236,4096")
    ap.add_argument("--check-rows", type=int, default=512)
    ap.add_argument("--kernel-time", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.kernel_time:
        return kernel_time(args)

    import torch

    from tools_b200 import _ffi

    info = gpu_info()
    T, gp, s, psf, a, td = setup()
    n, q, m, B = gp.n, gp.q, gp.m, args.batch
    ctx = psf.ctx
    rng = np.random.default_rng(1)
    sizes = [int(x) for x in args.tables.split(",")]
    tables = {t: unitriangular_tags(rng, t, n, q) for t in sizes}

    dev = torch.device("cuda", 0)
    tstream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(tstream)
    lib = _ffi.lib()
    ctx.call("qf_set_stream", _ffi.ptr(tstream.cuda_stream))
    u = torch.empty((B, n), dtype=torch.int64, device=dev)
    e = torch.empty((B, m), dtype=torch.int32, device=dev)
    idx_dev = {t: torch.from_numpy(rng.permutation(np.arange(B) % t).astype(np.int32)).to(dev) for t in sizes}
    check = Checker(gp, a, args.check_rows)
    install_s = {t: [] for t in sizes}

    def fill(i):
        assert lib.qf_fill_uniform_modq_dev(_ffi.ptr(u.data_ptr()), u.numel(), q, 1000 + i, _ffi.ptr(tstream.cuda_stream)) == 0

    def run(name, step):
        if name == "identity":
            ctx.call("qf_samp_p_dev", _ffi.ptr(u.data_ptr()), B, 2, step * B, _ffi.ptr(e.data_ptr()))
        else:
            ctx.call("qf_samp_p_tagged_dev", _ffi.ptr(u.data_ptr()), _ffi.ptr(idx_dev[name].data_ptr()), B, 2, step * B,
                     _ffi.ptr(e.data_ptr()))

    variants = ["identity"] + sizes
    rates = {str(k): [] for k in variants}
    for rnd in range(args.rounds):
        for name in variants:
            if name != "identity":
                tg = tables[name]
                install_s[name].append(sync_time(lambda: ctx.call("qf_set_tag_table", _ffi.ptr(tg), tg.shape[0])))
            for w in range(args.warmup):
                fill(w)
                run(name, w)
            ctx.call("qf_synchronize")
            ms = 0.0
            for k in range(args.steps):
                fill(args.warmup + k)
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ev0.record()
                run(name, args.warmup + k)
                ev1.record()
                ctx.call("qf_synchronize")
                ms += ev0.elapsed_time(ev1)
                check(e, u, idx_dev.get(name), tables.get(name), 100 * rnd + k)
            rates[str(name)].append(args.steps * B / (ms * 1e-3))
            print(f"round {rnd} {name}: {rates[str(name)][-1] / 1e6:.3f} M/s", file=sys.stderr)
    ctx.call("qf_set_stream", None)
    torch.cuda.set_stream(torch.cuda.default_stream(dev))
    del e, u
    torch.cuda.empty_cache()

    # ---- tag switch: qf_gpv_set_tag without / with the new basis, against qf_set_a + qf_set_trapdoor_gpv of that key
    h1, h2 = unitriangular_tags(rng, 2, n, q)
    a_new = np.empty((n, m), dtype=np.int64)
    s_new = np.empty((m, m), dtype=np.int64)
    switch_s, switch_basis_s, reinstall_s = [], [], []
    for rep in range(2):
        switch_s.append(sync_time(lambda: ctx.call("qf_gpv_set_tag", _ffi.ptr(h1), _ffi.ptr(a_new), None)))
        switch_basis_s.append(sync_time(lambda: ctx.call("qf_gpv_set_tag", _ffi.ptr(h2), _ffi.ptr(a_new), _ffi.ptr(s_new))))
    # a_new, s_new: the key and basis of H_2, installed from scratch as a caller without the switch would
    reinstall_s.append(sync_time(lambda: (ctx.call("qf_set_a", _ffi.ptr(a_new)),
                                          ctx.call("qf_set_trapdoor_gpv", _ffi.ptr(s_new), None),
                                          ctx.call("qf_synchronize"))))
    assert ctx.status("qf_set_tag_table", _ffi.ptr(tables[sizes[0]]), sizes[0]) == _ffi.QF_OK  # still two-phase

    best = {k: max(v) for k, v in rates.items()}
    res = {
        "metric": "PSFGPV samp_p targets/s with a tag per target (qf_samp_p_tagged_dev) vs the identity key (qf_samp_p_dev)",
        "workload": f"C2 PSFGPV n={n} q={q} m={m} s={s}, two-phase recursion, device-resident",
        "gpu": info,
        "batch_per_step": B, "warmup_steps": args.warmup, "timed_steps": args.steps, "rounds": args.rounds,
        "rates_per_round": rates,
        "best": best,
        "over_identity": {k: best[k] / best["identity"] for k in best if k != "identity"},
        "set_tag_table_s": {str(k): v for k, v in install_s.items()},
        "gpv_set_tag_s": switch_s,
        "gpv_set_tag_with_basis_s": switch_basis_s,
        "set_a_plus_set_trapdoor_gpv_s": reinstall_s,
        "verified_rows": check.checked,
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


def kernel_time(args):
    """torch.profiler (CUDA activities) over tagged steps with T = 236: time of the per-target tag kernel per step."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    from tools_b200 import _ffi

    info = gpu_info()
    T, gp, s, psf, a, td = setup()
    n, q, m, B = gp.n, gp.q, gp.m, args.batch
    ctx = psf.ctx
    rng = np.random.default_rng(1)
    tags = unitriangular_tags(rng, 236, n, q)
    ctx.call("qf_set_tag_table", _ffi.ptr(tags), 236)
    dev = torch.device("cuda", 0)
    u = torch.empty((B, n), dtype=torch.int64, device=dev)
    e = torch.empty((B, m), dtype=torch.int32, device=dev)
    idx = torch.from_numpy(rng.permutation(np.arange(B) % 236).astype(np.int32)).to(dev)
    lib = _ffi.lib()
    assert lib.qf_fill_uniform_modq_dev(_ffi.ptr(u.data_ptr()), u.numel(), q, 5, None) == 0
    torch.cuda.synchronize()
    for w in range(args.warmup):
        ctx.call("qf_samp_p_tagged_dev", _ffi.ptr(u.data_ptr()), _ffi.ptr(idx.data_ptr()), B, 2, w * B, _ffi.ptr(e.data_ptr()))
    ctx.call("qf_synchronize")
    res = None
    for attempt in range(2):  # an empty capture is retried once
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for k in range(args.steps):
                ctx.call("qf_samp_p_tagged_dev", _ffi.ptr(u.data_ptr()), _ffi.ptr(idx.data_ptr()), B, 2, k * B,
                         _ffi.ptr(e.data_ptr()))
            ctx.call("qf_synchronize")
        tot, cnt, all_us = 0.0, 0, 0.0
        for ev in prof.key_averages():
            us = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
            all_us += us
            if "tag_syndrome" in ev.key:
                tot += us
                cnt += ev.count
        if cnt:
            res = {"metric": "per-target tag kernel time per step (torch.profiler, CUDA activities)", "gpu": info,
                   "workload": f"C2 PSFGPV n={n} q={q} m={m} T=236 batch={B}", "steps": args.steps, "launches": cnt,
                   "tag_kernel_ms_per_step": tot / 1e3 / args.steps, "all_kernels_ms_per_step": all_us / 1e3 / args.steps}
            break
    if res is None:
        res = {"metric": "per-target tag kernel time per step", "gpu": info, "not_measured": "profiler captured no tag kernel"}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
