"""samp_p with a tag per target (qf_set_tag_table + qf_samp_p_tagged_dev, DESIGN.md 4.4) against the plain identity key.

One C4 shard (PSFPerturbation n = 512, q = 2^32 - 5, m = 32849, r = 9, structured sqrt(Sigma_2)), device-resident, 60 416
targets per step (bench.py c4), 3 warm-up and 4 timed steps per variant (CUDA events), the variants alternating in each of
two rounds on one context:
  identity   qf_samp_p_dev on the identity key A = [A_bar | G - A_bar R]
  T=1        qf_samp_p_tagged_dev with a table of one tag
  T=236      236 tags (256 targets per tag)
  T=4096     4096 tags (about 15 targets per tag)
Tags are random upper unitriangular, tag indices shuffled.  On every timed output A_t e = u is checked exactly on a seeded
sample of 512 rows on the host (16-bit splits in float64: A_t e = A e + (H_t - I) G e_bot).  Also times qf_set_tag_table for
T = 236 and 4096 (host clock around the synchronised call), and for 8 192 targets under 32 tags the tagged call against
what a caller does without the table: 32 x (qf_set_tag + qf_samp_p_dev on that tag's rows).  Prints one JSON line, with the
card name and power limit.

  python scripts/bench_tag_table.py [--out FILE]
  python scripts/bench_tag_table.py --kernel-time   # a run of its own: torch.profiler (CUDA activities) time of the
                                                    # per-target tag kernel per step
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


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in out.split(",")]
    return {"name": name, "power_limit": power}


def unitriangular_tags(rng, count, n, q):
    """count random upper unitriangular n x n tags, built in place (4096 tags at n = 512 are 8 GB of int64)."""
    t = rng.integers(0, q, (count, n, n), dtype=np.int64)
    t *= np.triu(np.ones((n, n), dtype=np.int64), 1)
    t += np.eye(n, dtype=np.int64)
    return t


def mulmod16(x, y, q):
    """x y mod q for int64 residues < 2^32 (x: B x K, y: K x N), exact with 16-bit halves in float64 (K < 2^20)."""
    x0, x1 = (x & 0xFFFF).astype(np.float64), (x >> 16).astype(np.float64)
    y0, y1 = (y & 0xFFFF).astype(np.float64), (y >> 16).astype(np.float64)
    p00 = np.rint(x0 @ y0).astype(np.int64) % q
    p01 = (np.rint(x0 @ y1).astype(np.int64) + np.rint(x1 @ y0).astype(np.int64)) % q
    p11 = np.rint(x1 @ y1).astype(np.int64) % q
    return (p00 + (p01 << 16) % q + (((p11 << 16) % q) << 16) % q) % q


class Checker:
    """A_t e = u on a seeded sample of rows: A e (16-bit halves of A, |e| < 2^16) plus (H_t - I) y, y = G e_bot mod q."""

    def __init__(self, gp, a, rows):
        self.gp, self.rows = gp, rows
        self.a_lo = (a & 0xFFFF).astype(np.float64).T.copy()
        self.a_hi = (a >> 16).astype(np.float64).T.copy()
        self.gpow = np.array([gp.base**s % gp.q for s in range(gp.k)], dtype=np.int64)
        self.checked = 0

    def __call__(self, e_dev, u_dev, idx_dev, tags, seed):
        gp, q = self.gp, self.gp.q
        sel = np.sort(np.random.default_rng(seed).choice(e_dev.shape[0], self.rows, replace=False))
        import torch

        ti = torch.from_numpy(sel).to(e_dev.device)
        e = e_dev.index_select(0, ti).cpu().numpy()
        u = u_dev.index_select(0, ti).cpu().numpy()
        ef = e.astype(np.float64)
        ae = (np.rint(ef @ self.a_lo).astype(np.int64) % q + ((np.rint(ef @ self.a_hi).astype(np.int64) % q) << 16) % q) % q
        if tags is not None:
            idx = idx_dev.index_select(0, ti).cpu().numpy()
            eb = e[:, gp.m_bar:].astype(np.int64).reshape(len(e), gp.n, gp.k) % q
            y = mulmod16(eb.reshape(-1, gp.k), self.gpow.reshape(-1, 1), q).reshape(len(e), gp.n)
            for b in range(len(e)):
                d = tags[idx[b]].copy()
                d[np.arange(gp.n), np.arange(gp.n)] -= 1
                ae[b] = (ae[b] + mulmod16(y[b:b + 1], (d % q).T, q)[0]) % q
        assert np.array_equal(ae, u), "A_t e != u"
        self.checked += len(e)


def setup(args):
    import tools_b200 as T

    n, q, r = args.n, args.q, 9.0
    gp = T.GadgetParameters.init_default(n, q)
    s1 = (math.sqrt(gp.m_bar) + math.sqrt(n * gp.k)) / math.sqrt(2)
    s = float(math.ceil(1.15 * math.sqrt(5 * (s1 * s1 + 1) + 1)))  # bench.py pert_s_for
    psf = T.PSFPerturbation(gp, r, s)
    a, td = psf.trap_gen(seed=2, dense_sqrt_sigma_2=False)
    psf._install_a(a)
    psf._install_td(a, td)
    return T, gp, r, s, psf, a, td


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--q", type=int, default=2**32 - 5)
    ap.add_argument("--batch", type=int, default=60416)
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
    T, gp, r, s, psf, a, td = setup(args)
    n, q, m, B = gp.n, gp.q, gp.m, args.batch
    ctx = psf.ctx
    rng = np.random.default_rng(1)
    sizes = [int(x) for x in args.tables.split(",")]
    tables = {t: unitriangular_tags(rng, t, n, q) for t in sizes}

    def sync_time(f):
        t0 = time.time()
        f()
        return time.time() - t0

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
            print(f"round {rnd} {name}: {rates[str(name)][-1] / 1e3:.1f} k/s", file=sys.stderr)

    # ---- 8 192 targets under 32 tags: one tagged call against 32 x (qf_set_tag + qf_samp_p_dev on that tag's rows)
    B2, T2 = 8192, 32
    tags32 = unitriangular_tags(rng, T2, n, q)
    idx32 = rng.permutation(np.arange(B2) % T2).astype(np.int32)
    fill(77)
    u2 = u[:B2].clone()
    e2 = torch.empty((B2, m), dtype=torch.int32, device=dev)
    i2 = torch.from_numpy(idx32).to(dev)
    ctx.call("qf_set_tag_table", _ffi.ptr(tags32), T2)
    ctx.call("qf_samp_p_tagged_dev", _ffi.ptr(u2.data_ptr()), _ffi.ptr(i2.data_ptr()), B2, 3, 0, _ffi.ptr(e2.data_ptr()))
    ctx.call("qf_synchronize")  # warm
    tagged_s = []
    for rep in range(2):
        torch.cuda.synchronize()
        tagged_s.append(sync_time(lambda: (ctx.call("qf_samp_p_tagged_dev", _ffi.ptr(u2.data_ptr()), _ffi.ptr(i2.data_ptr()),
                                                    B2, 3, 0, _ffi.ptr(e2.data_ptr())), ctx.call("qf_synchronize"))))
    check(e2, u2, i2, tags32, 999)
    groups = [torch.from_numpy(np.flatnonzero(idx32 == t)).to(dev) for t in range(T2)]
    ug = [u2.index_select(0, g).contiguous() for g in groups]
    eg = [torch.empty((len(g), m), dtype=torch.int32, device=dev) for g in groups]
    torch.cuda.synchronize()

    def per_tag_loop():
        cur = a
        for t in range(T2):
            cur = psf.set_tag(cur, td, tags32[t])
            ctx.call("qf_samp_p_dev", _ffi.ptr(ug[t].data_ptr()), ug[t].shape[0], 3, 0, _ffi.ptr(eg[t].data_ptr()))
        ctx.call("qf_synchronize")
        return cur

    loop_s = []
    holder = {}
    loop_s.append(sync_time(lambda: holder.setdefault("a", per_tag_loop())))
    # back to the identity key (untimed) so that the context ends as it started
    psf.set_tag(holder["a"], td, None)
    ctx.call("qf_set_stream", None)
    torch.cuda.set_stream(torch.cuda.default_stream(dev))

    best = {k: max(v) for k, v in rates.items()}
    res = {
        "metric": "samp_p targets/s with a tag per target (qf_samp_p_tagged_dev) vs the identity key (qf_samp_p_dev)",
        "workload": f"PSFPerturbation n={n} q={q} m={m} r={r} s={s} structured sqrt(Sigma_2), one C4 shard",
        "gpu": info,
        "batch_per_step": B, "warmup_steps": args.warmup, "timed_steps": args.steps, "rounds": args.rounds,
        "rates_per_round": rates,
        "best": best,
        "over_identity": {k: best[k] / best["identity"] for k in best if k != "identity"},
        "set_tag_table_s": {str(k): v for k, v in install_s.items()},
        "mixed_8192_targets_32_tags": {"tagged_call_s": tagged_s, "set_tag_plus_samp_p_loop_s": loop_s,
                                       "speedup": min(loop_s) / min(tagged_s)},
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
    T, gp, r, s, psf, a, td = setup(args)
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
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for k in range(args.steps):
            ctx.call("qf_samp_p_tagged_dev", _ffi.ptr(u.data_ptr()), _ffi.ptr(idx.data_ptr()), B, 2, k * B, _ffi.ptr(e.data_ptr()))
        ctx.call("qf_synchronize")
    tot, cnt, all_us = 0.0, 0, 0.0
    for ev in prof.key_averages():
        us = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        all_us += us
        if "tag_syndrome" in ev.key:
            tot += us
            cnt += ev.count
    res = {"metric": "per-target tag kernel time per step (torch.profiler, CUDA activities)", "gpu": info,
           "workload": f"n={n} q={q} m={m} T=236 batch={B}", "steps": args.steps, "launches": cnt,
           "tag_kernel_ms_per_step": tot / 1e3 / args.steps, "all_kernels_ms_per_step": all_us / 1e3 / args.steps}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
