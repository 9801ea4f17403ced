"""f_a with a tag per target (qf_set_f_a_tags + qf_f_a_tagged_dev, DESIGN.md 4.9) against untagged f_a.

Workloads (keys built from a uniform A_bar and a random R with H_0 = I; the context holds only the key):
  C2   PSFGPV n = 256, q = 2^24, m = 12352, 65 536 targets per pass (3.2 GB of sigma)
  C4   one PSFPerturbation shard n = 512, q = 2^32 - 5, m = 32849, 15 104 targets per pass (2.0 GB of sigma)
sigma comes from qf_samp_d_dev and stays on the device; it is far larger than the 126 MB L2.  Variants, alternating in each
of two rounds on one context: qf_f_a_dev (untagged) and qf_f_a_tagged_dev with T = 1, 236 and 4096 random dense tags and
shuffled tag indices.  Per variant 3 warm-up passes, then enough timed passes for about one second (CUDA events).  Every
timed output is checked exactly: a seeded sample of 64 rows against the CPU (16-bit halves in float64), and every
in_domain flag.  In the same run: torch.profiler (CUDA activities) times of the sort kernels and of the correction kernel,
qf_set_f_a_tags install times, and the same measurement with the library rebuilt at QF_F_A_TAG_GROUP = 1 (one target per
CTA, no sort) in a temporary directory.  Writes one JSON file with the card name and power limit.

  python scripts/bench_f_a_tagged.py [--out FILE] [--quick]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = {"c2": dict(kind="gpv", n=256, q=2**24, batch=65536), "c4": dict(kind="pert", n=512, q=2**32 - 5, batch=15104)}
TAG_COUNTS = (1, 236, 4096)
SAMPLE = 64


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in out.split(",")]
    return {"name": name, "power_limit": power}


def build_group1(tmp):
    """the library with QF_F_A_TAG_GROUP = 1, every source compiled into tmp"""
    from tools_b200 import build as B

    objs, procs = [], []
    for s in B.SOURCES:
        o = os.path.join(tmp, s.replace(".cu", ".o"))
        cmd = [B._nvcc()] + B.NVCC_FLAGS + ["-DQF_F_A_TAG_GROUP=1", "-c", os.path.join(B.CSRC, s), "-o", o]
        procs.append(subprocess.Popen(cmd))
        objs.append(o)
    if any(p.wait() for p in procs):
        raise SystemExit("nvcc failed on the QF_F_A_TAG_GROUP = 1 build")
    lib = os.path.join(tmp, "libqfall_b200.so")
    subprocess.check_call([B._nvcc(), "-shared", "-o", lib] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "shared"])
    return lib


def mm(x, y, q):
    """x @ y mod q exactly for int64 |x| < 2^32, y in [0, q), q <= 2^32 (16-bit halves in float64)"""
    x0, x1 = (x & 0xFFFF).astype(np.float64), (x >> 16).astype(np.float64)
    y0, y1 = (y & 0xFFFF).astype(np.float64), (y >> 16).astype(np.float64)
    r = lambda a, b: np.rint(a @ b).astype(np.int64) % q  # noqa: E731
    s16 = (1 << 16) % q
    return (r(x0, y0) + (r(x0, y1) + r(x1, y0)) % q * s16 % q + r(x1, y1) * s16 % q * s16 % q) % q


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def run(quick):
    import torch
    from tools_b200 import _ffi, gadget, psf as P

    dev = torch.device("cuda:0")
    res = {}
    for wname, w in WORKLOADS.items():
        n, q, batch = w["n"], w["q"], w["batch"] // (16 if quick else 1)
        gp = gadget.GadgetParameters.init_default(n, q)
        kind = _ffi.QF_PSF_GPV if w["kind"] == "gpv" else _ffi.QF_PSF_PERTURBATION
        ctx = _ffi.Context(kind, n, gp.k, gp.m_bar, gp.base, q, 300.0, 9.0, 0)
        ctx.call("qf_set_stream", _ffi.ptr(torch.cuda.current_stream().cuda_stream))  # the events time the library's work
        rng = np.random.default_rng(n)
        a_bar = rng.integers(0, q, (n, gp.m_bar), dtype=np.int64)
        r = rng.integers(-1, 2, (gp.m_bar, n * gp.k)).astype(np.int8)
        a = P.gen_trapdoor(gp, a_bar, r)
        ctx.call("qf_set_a", _ffi.ptr(np.ascontiguousarray(a)))
        m = gp.m
        sig = torch.empty((batch, m), dtype=torch.int32, device=dev)
        ctx.call("qf_samp_d_dev", batch, 5, 0, _ffi.ptr(sig.data_ptr()))
        ctx.call("qf_synchronize")
        u = torch.empty((batch, n), dtype=torch.int64, device=dev)
        fl = torch.empty(batch, dtype=torch.uint8, device=dev)
        rows = np.sort(np.random.default_rng(7).choice(batch, SAMPLE, replace=False))
        s_rows = sig[torch.from_numpy(rows).to(dev)].cpu().numpy().astype(np.int64)
        au = mm(s_rows, a.T, q)
        gpow = np.array([pow(gp.base, s, q) for s in range(gp.k)], dtype=np.int64).reshape(-1, 1)
        y = mm(s_rows[:, gp.m_bar:].reshape(-1, gp.k), gpow, q).reshape(SAMPLE, n)
        tables = {}
        log(wname, "sigma ready")
        out = {"n": n, "q": q, "m": m, "batch": batch, "install_s": {}, "rate_per_s": {}, "kernel_ms_per_pass": {}}
        for T in TAG_COUNTS:
            tt = min(T, 16) if quick else T
            tags = rng.integers(0, q, (tt, n, n), dtype=np.int64)
            idx = torch.from_numpy(rng.permutation(np.arange(batch) % tt).astype(np.int32)).to(dev)
            t0 = time.perf_counter()
            ctx.call("qf_set_f_a_tags", _ffi.ptr(tags), tt, None)
            out["install_s"][f"T={T}"] = time.perf_counter() - t0
            log(wname, f"T={T} installed in {out['install_s'][f'T={T}']:.2f} s")
            want = au.copy()
            ic = idx[torch.from_numpy(rows).to(dev)].cpu().numpy()
            for i in range(SAMPLE):
                d = (tags[ic[i]] - np.eye(n, dtype=np.int64)) % q
                want[i] = (want[i] + mm(y[i:i + 1], d.T, q)[0]) % q
            tables[T] = (tags, idx, want)
        cur = [None]

        def use(T):  # one table on the device at a time (4096 tags at C4 are 4 GB)
            if cur[0] != T:
                ctx.call("qf_set_f_a_tags", _ffi.ptr(tables[T][0]), len(tables[T][0]), None)
                cur[0] = T

        def call(T):
            if T is None:
                ctx.call("qf_f_a_dev", _ffi.ptr(sig.data_ptr()), batch, _ffi.ptr(u.data_ptr()), _ffi.ptr(fl.data_ptr()))
            else:
                ctx.call("qf_f_a_tagged_dev", _ffi.ptr(sig.data_ptr()), _ffi.ptr(tables[T][1].data_ptr()), batch,
                         _ffi.ptr(u.data_ptr()), _ffi.ptr(fl.data_ptr()))

        def check(T):
            ctx.call("qf_synchronize")
            got = u[torch.from_numpy(rows).to(dev)].cpu().numpy()
            want = au if T is None else tables[T][2]
            assert np.array_equal(got, want), (wname, T)
            assert bool(fl.bool().all()), (wname, T)

        variants = [None] + list(TAG_COUNTS)
        rates = {str(v): [] for v in variants}
        for _ in range(2):
            for T in variants:
                if T is not None:
                    use(T)
                for _ in range(3):
                    call(T)
                ctx.call("qf_synchronize")
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                call(T)
                e1.record()
                e1.synchronize()
                reps = max(3, min(5000, int(1000.0 / max(e0.elapsed_time(e1), 1e-3))))
                if quick:
                    reps = 3
                e0.record()
                for _ in range(reps):
                    call(T)
                e1.record()
                e1.synchronize()
                rates[str(T)].append(batch * reps / (e0.elapsed_time(e1) / 1e3))
                check(T)
                log(wname, T, f"{rates[str(T)][-1]:.4g} targets/s")
        out["rate_per_s"] = {("untagged" if k == "None" else f"T={k}"): v for k, v in rates.items()}
        # kernel times: a profiled pass of its own per variant
        from torch.profiler import ProfilerActivity, profile

        def kernel_times(T):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(5):
                    call(T)
                ctx.call("qf_synchronize")
            ks = {}
            for ev in prof.key_averages():
                name = ev.key
                tag = ("sort_hist" if "fa_tag_hist" in name else "sort_scan" if "fa_tag_scan" in name else
                       "sort_scatter" if "fa_tag_scatter" in name else "correct" if "fa_tag_correct" in name else
                       "f_a" if "f_a_fused" in name or "gemm" in name or "split" in name or "domain_flags" in name else
                       "memset" if "emset" in name else None)
                if tag and ev.device_time_total > 0:
                    ks[tag] = ks.get(tag, 0.0) + ev.device_time_total / 1e3 / 5
            return ks

        out["not_measured"] = []
        for T in variants:
            if T is not None:
                use(T)
            call(T)
            ctx.call("qf_synchronize")
            name = "untagged" if T is None else f"T={T}"
            need = ("f_a",) if T is None else ("f_a", "correct")
            for _ in range(3):  # a profiler session now and then records no kernels: try again, then say so
                ks = kernel_times(T)
                if all(k in ks for k in need):
                    break
            missing = [k for k in need if k not in ks]
            if missing:
                log(f"WARNING {wname} {name}: the profiler recorded no {', '.join(missing)} kernel; not measured")
                out["not_measured"].append(f"{name}: {', '.join(missing)}")
            out["kernel_ms_per_pass"][name] = ks
        res[wname] = out
        del sig, u, fl, tables
        ctx.call("qf_set_stream", None)
        ctx.close()
        torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_f_a_tagged.json"))
    ap.add_argument("--quick", action="store_true", help="small batches and tables: a smoke run of the script")
    ap.add_argument("--lib", help=argparse.SUPPRESS)  # run against another build of the library (the QF_F_A_TAG_GROUP = 1 pass)
    args = ap.parse_args()
    if args.lib:
        from tools_b200 import _ffi

        _ffi.LIB_PATH = args.lib
        print(json.dumps(run(args.quick)))
        return
    from tools_b200 import build as B

    B.build()
    info = gpu_info()
    grouped = run(args.quick)
    with tempfile.TemporaryDirectory() as tmp:
        lib = build_group1(tmp)
        cmd = [sys.executable, os.path.abspath(__file__), "--lib", lib] + (["--quick"] if args.quick else [])
        p = subprocess.run(cmd, stdout=subprocess.PIPE, text=True)
        if p.returncode:
            raise SystemExit("the QF_F_A_TAG_GROUP = 1 pass failed")
        g1 = json.loads(p.stdout.strip().splitlines()[-1])
    result = {"gpu": info, "group": 8, "grouped": grouped, "group_1_no_sort": g1,
              "note": "rate_per_s: targets/s of device-resident f_a, one value per alternating round; summary: their mean; "
                      "kernel_ms_per_pass: torch.profiler CUDA time per pass"}
    for w in grouped:
        result.setdefault("summary", {})[w] = {
            k: {"grouped": float(np.mean(v)), "group_1": float(np.mean(g1[w]["rate_per_s"][k])),
                "vs_untagged": float(np.mean(v) / np.mean(grouped[w]["rate_per_s"]["untagged"]))}
            for k, v in grouped[w]["rate_per_s"].items()}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["summary"]))
    for run_name, r in (("grouped", grouped), ("group_1_no_sort", g1)):
        for w in r:
            if r[w]["not_measured"]:
                print(f"not measured ({run_name}, {w}): {r[w]['not_measured']}", file=sys.stderr)
    print(json.dumps(info))


if __name__ == "__main__":
    main()
