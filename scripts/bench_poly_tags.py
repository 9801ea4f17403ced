"""Tags in polynomial form (qf_set_tag_table_poly, qf_set_f_a_tags_poly; DESIGN.md 4.10) against the matrix tag tables.

Two workloads, device-resident targets, tags h_t random in Z_q[X]/(X^n + 1) (for q = 2^24 made units by h(1) odd), the
matrix tags H_t = rot_f(h_t) built from the same h_t:
  c4  one C4 shard: PSFPerturbation n = 512, q = 2^32 - 5, m = 32849, r = 9, structured sqrt(Sigma_2), 60 416 targets
  c2  PSFGPV n = 256, q = 2^24, m = 12352 on the two-phase recursion, 37 888 targets
Measured per workload (host clock around work that ends in a device synchronise):
  install   qf_set_tag_table (matrix) and qf_set_tag_table_poly for T = 236 and 4096, and T = 65 536 polynomial only
  samp_p    qf_samp_p_dev on the identity key, qf_samp_p_tagged_dev with the matrix and polynomial tables of T = 236 and
            4096, and with one polynomial tag per target; variants alternate within each round
  f_a       qf_f_a_tagged_dev with the matrix and the polynomial f_a table of T = 4096 (sigma = a sampled step)
  fresh     B = 4096 targets under B distinct new tags: install plus one sampling call, matrix against polynomial
Every timed samp_p output is checked: A_t e = u exactly on a seeded sample of rows, evaluated by qf_f_a_tagged_dev with a
polynomial f_a table of the same tags (H_t = rot_f(h_t); the identity key as the tag h = 1).  Prints one JSON line with
the card name and power limit read in the same run.

  python scripts/bench_poly_tags.py [--workloads c4,c2] [--out FILE]
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


def negacyclic(h, q):
    """rot_f(h) for f = X^n + 1 of T tags at once (T x n x n int64, mod q): column c is h X^c mod X^n + 1."""
    t, n = h.shape
    i = np.arange(n)[:, None]
    c = np.arange(n)[None, :]
    src = (i - c) % n
    out = h[:, src]
    out[:, i < c] *= -1  # broadcast over the wrapped entries
    out %= q
    return out


def poly_tags(rng, count, n, q):
    h = rng.integers(0, q, (count, n), dtype=np.int64)
    if q % 2 == 0:  # X^n + 1 = (X + 1)^n mod 2: h is a unit iff h(1) is odd
        h[:, 0] += (h.sum(axis=1) + 1) % 2
    return h


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
        B = 37888
    psf._install_a(a)
    psf._install_td(a, td)
    return gp, psf, a, td, B


def run_workload(T, name, args):
    import torch

    from tools_b200 import _ffi

    gp, psf, a, td, B = setup(T, name)
    n, q, m = gp.n, gp.q, gp.m
    ctx = psf.ctx
    rng = np.random.default_rng(7)
    f = np.array([1] + [0] * (n - 1), dtype=np.int64)
    fw = np.ascontiguousarray(f)
    dev = torch.device("cuda", 0)
    res = {"n": n, "q": q, "m": m, "targets_per_step": B}

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.time()
        fn()
        ctx.call("qf_synchronize")
        torch.cuda.synchronize()
        return time.time() - t0

    # ---- install times
    hs = {t: poly_tags(rng, t, n, q) for t in (236, 4096)}
    hs[B] = poly_tags(rng, B, n, q)  # one tag per target
    mats = {t: np.ascontiguousarray(negacyclic(hs[t], q)) for t in (236, 4096)}
    inst = {}
    for t in (236, 4096):
        inst[f"matrix_T{t}_s"] = timed(lambda: ctx.call("qf_set_tag_table", _ffi.ptr(mats[t]), t))
        ht = np.ascontiguousarray(hs[t])
        inst[f"poly_T{t}_s"] = timed(lambda: ctx.call("qf_set_tag_table_poly", _ffi.ptr(fw), _ffi.ptr(ht), t))
    h64 = np.ascontiguousarray(poly_tags(rng, 65536, n, q))
    inst["poly_T65536_s"] = timed(lambda: ctx.call("qf_set_tag_table_poly", _ffi.ptr(fw), _ffi.ptr(h64), 65536))
    del h64
    res["install"] = inst

    # ---- samp_p rates
    u = torch.randint(0, q, (B, n), dtype=torch.int64, device=dev)
    e = torch.empty((B, m), dtype=torch.int32, device=dev)
    idx = {t: torch.from_numpy((np.arange(B) % t)[rng.permutation(B)].astype(np.int32)).to(dev) for t in (236, 4096, B)}

    def install(kind, t):
        if kind == "matrix":
            ctx.call("qf_set_tag_table", _ffi.ptr(mats[t]), t)
        elif kind == "poly":
            ht = np.ascontiguousarray(hs[t])
            ctx.call("qf_set_tag_table_poly", _ffi.ptr(fw), _ffi.ptr(ht), t)

    def step(kind, t, seed):
        if kind == "identity":
            ctx.call("qf_samp_p_dev", _ffi.ptr(u.data_ptr()), B, seed, 0, _ffi.ptr(e.data_ptr()))
        else:
            ctx.call("qf_samp_p_tagged_dev", _ffi.ptr(u.data_ptr()), _ffi.ptr(idx[t].data_ptr()), B, seed, 0,
                     _ffi.ptr(e.data_ptr()))

    checked = [0]
    ones = np.zeros((1, n), dtype=np.int64)
    ones[0, 0] = 1

    def check(kind, t, seed):
        sel = torch.from_numpy(np.sort(np.random.default_rng(seed).choice(B, args.check_rows, replace=False))).to(dev)
        es, us = e.index_select(0, sel).contiguous(), u.index_select(0, sel)
        if kind == "identity":
            ht, ti = ones, torch.zeros(len(sel), dtype=torch.int32, device=dev)
        else:
            ht, ti = np.ascontiguousarray(hs[t]), idx[t].index_select(0, sel).contiguous()
        ctx.call("qf_set_f_a_tags_poly", _ffi.ptr(fw), _ffi.ptr(ht), len(ht), None)
        got = torch.empty_like(us)
        ok = torch.empty(len(sel), dtype=torch.uint8, device=dev)
        ctx.call("qf_f_a_tagged_dev", _ffi.ptr(es.data_ptr()), _ffi.ptr(ti.data_ptr()), len(sel), _ffi.ptr(got.data_ptr()),
                 _ffi.ptr(ok.data_ptr()))
        ctx.call("qf_synchronize")
        assert torch.equal(got, us) and bool(ok.all()), (name, kind, t)
        checked[0] += len(sel)

    variants = [("identity", 0), ("matrix", 236), ("poly", 236), ("matrix", 4096), ("poly", 4096), ("poly", B)]
    times = {f"{k}_T{t}" if t else k: [] for k, t in variants}
    for rnd in range(args.rounds):
        for kind, t in variants:
            key = f"{kind}_T{t}" if t else kind
            install(kind, t)
            for w in range(args.warmup):
                step(kind, t, 100 + w)
            ctx.call("qf_synchronize")
            torch.cuda.synchronize()
            times[key].append(timed(lambda: [step(kind, t, 1000 * rnd + s) for s in range(args.steps)]) / args.steps)
            check(kind, t, 1000 * rnd + args.steps - 1)
    res["samp_p_targets_per_s"] = {k: B / min(v) for k, v in times.items()}
    res["samp_p_step_s"] = {k: sorted(v) for k, v in times.items()}

    # ---- f_a rates at T = 4096 on the last sampled step (sigma = e)
    t = 4096
    install("poly", t)
    step("poly", t, 7)
    got = torch.empty_like(u)
    ok = torch.empty(B, dtype=torch.uint8, device=dev)
    fa = {}
    h4 = np.ascontiguousarray(hs[t])
    for rnd in range(args.rounds):
        for kind in ("matrix", "poly"):
            if kind == "matrix":
                ctx.call("qf_set_f_a_tags", _ffi.ptr(mats[t]), t, None)
            else:
                ctx.call("qf_set_f_a_tags_poly", _ffi.ptr(fw), _ffi.ptr(h4), t, None)

            def call():
                ctx.call("qf_f_a_tagged_dev", _ffi.ptr(e.data_ptr()), _ffi.ptr(idx[t].data_ptr()), B,
                         _ffi.ptr(got.data_ptr()), _ffi.ptr(ok.data_ptr()))

            for _ in range(args.warmup):
                call()
            ctx.call("qf_synchronize")
            torch.cuda.synchronize()
            fa.setdefault(kind, []).append(timed(lambda: [call() for _ in range(args.steps)]) / args.steps)
            assert torch.equal(got, u) and bool(ok.all()), (name, "f_a", kind)
    res["f_a_T4096_targets_per_s"] = {k: B / min(v) for k, v in fa.items()}

    # ---- fresh identities: B' targets under B' new tags, install + one sampling call
    Bf = 4096
    hf = np.ascontiguousarray(poly_tags(rng, Bf, n, q))
    mf = np.ascontiguousarray(negacyclic(hf, q))
    uf = u[:Bf].contiguous()
    ef = e[:Bf]
    idf = torch.from_numpy(rng.permutation(Bf).astype(np.int32)).to(dev)
    fresh = {}
    for kind in ("matrix", "poly"):
        def run():
            if kind == "matrix":
                ctx.call("qf_set_tag_table", _ffi.ptr(mf), Bf)
            else:
                ctx.call("qf_set_tag_table_poly", _ffi.ptr(fw), _ffi.ptr(hf), Bf)
            ctx.call("qf_samp_p_tagged_dev", _ffi.ptr(uf.data_ptr()), _ffi.ptr(idf.data_ptr()), Bf, 5, 0, _ffi.ptr(ef.data_ptr()))
        fresh[f"{kind}_s"] = timed(run)
    res["fresh_4096_targets_4096_tags"] = fresh
    res["rows_checked"] = checked[0]
    del psf
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c4,c2")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--check-rows", type=int, default=256)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import tools_b200 as T

    line = {"gpu": gpu_info(), "steps": args.steps, "warmup": args.warmup, "rounds": args.rounds,
            "not_measured": ["kernel times (no profiler run)"]}
    for w in args.workloads.split(","):
        line[w] = run_workload(T, w, args)
    line["gpu_after"] = gpu_info()
    s = json.dumps(line)
    print(s, flush=True)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(s + "\n")


if __name__ == "__main__":
    main()
