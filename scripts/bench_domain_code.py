"""Packed preimages (qf_samp_p_packed, qf_f_a_packed; DESIGN.md 4.11) against the int16 host-buffer form.

Workloads, host targets and results in pinned host buffers:
  c2  PSFGPV n = 256, q = 2^24, m = 12352 on the two-phase recursion, 227 328 targets per call (six default chunks)
  c4  one C4 shard: PSFPerturbation n = 512, q = 2^32 - 5, m = 32849, r = 9, structured sqrt(Sigma_2), 60 416 targets
Measured per workload (host clock around calls that synchronise): qf_samp_p_i16 against qf_samp_p_packed at the
parameters of qf_domain_code_params, 3 warm-up calls each, then two rounds of 4 timed calls of each, alternated; the mean
and maximum nbytes seen; qf_f_a_i16 against qf_f_a_packed on the preimages of the last call (2 warm-up, 4 timed, alternated).
Every timed output is checked: a seeded sample of packed rows decoded on the device equals qf_samp_p at those indices, the
int16 rows equal the decoded ones, and f_a of both forms gives back u exactly (A e = u) with every row in the domain.
A separate run under torch.profiler gives the encode / decode kernel times for one default chunk.  Writes one JSON file
with the card name and power limit read in the same run.

  python scripts/bench_domain_code.py [--workloads c2,c4] [--out FILE]
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

# bytes per target of the packed form at w, from the Gaussian law (the issue table): C2, C4
EXPECTED_MEAN = {"c2": 17458, "c4": 52566}


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


def pinned(shape, dtype):
    import torch

    return torch.empty(shape, dtype=dtype, pin_memory=True).numpy()


def run_workload(T, name, args):
    import torch

    from tools_b200 import _ffi, domain_code

    gp, psf, a, td, B = setup(T, name)
    n, q, m = gp.n, gp.q, gp.m
    ctx = psf.ctx
    k, slot = psf.domain_code_params()
    u = pinned((B, n), torch.int64)
    u[:] = np.random.default_rng(7).integers(0, q, (B, n), dtype=np.int64)
    e16 = pinned((B, m), torch.int16)
    pk = pinned((B, slot), torch.uint8)
    nb = pinned((B,), torch.int32)
    res = {"n": n, "q": q, "m": m, "w": psf.s * (psf.r if name == "c4" else 1.0), "targets_per_call": B, "k": k,
           "slot_bytes": slot, "int16_bytes_per_target": 2 * m}

    def call_i16(seed):
        ctx.call("qf_samp_p_i16", _ffi.ptr(u), B, seed, 0, _ffi.ptr(e16))

    def call_packed(seed):
        st = ctx.status("qf_samp_p_packed", _ffi.ptr(u), None, B, seed, 0, k, slot, _ffi.ptr(pk), _ffi.ptr(nb))
        assert st in (_ffi.QF_OK, _ffi.QF_ERR_NUMERIC), st

    def timed(fn, seed):
        t0 = time.time()
        fn(seed)
        return time.time() - t0

    for i in range(3):
        call_i16(100 + i)
        call_packed(100 + i)
    times = {"int16": [], "packed": []}
    overflow_rows, nb_mean, nb_max = 0, [], 0
    for rnd in range(2):
        for fn, key in ((call_i16, "int16"), (call_packed, "packed")):
            for i in range(args.calls):
                seed = 1000 * rnd + i
                times[key].append(timed(fn, seed))
                if key == "packed":
                    overflow_rows += int((nb < 0).sum())
                    nb_mean.append(float(nb[nb >= 0].mean()))
                    nb_max = max(nb_max, int(nb.max()))
    # the last packed call used seed 1000 + calls - 1; the int16 call of that seed, then checks on both
    seed = 1000 + args.calls - 1
    call_i16(seed)
    rows = np.sort(np.random.default_rng(seed).choice(B, args.check_rows, replace=False))
    dec, ok = domain_code.decode(torch.from_numpy(pk[rows]).cuda(), m, k)
    dec, ok = dec.cpu().numpy(), ok.cpu().numpy()
    assert ok.all()
    for j, b in enumerate(rows):
        e1 = np.empty((1, m), dtype=np.int32)
        ctx.call("qf_samp_p", _ffi.ptr(np.ascontiguousarray(u[b:b + 1])), 1, seed, int(b), _ffi.ptr(e1))
        assert np.array_equal(e1[0], dec[j]), (name, b)
        assert np.array_equal(e16[b].astype(np.int32), dec[j]), (name, b)
    # f_a of both forms on these preimages: A e = u, every row in the domain
    uo = pinned((B, n), torch.int64)
    fl = pinned((B,), torch.uint8)

    def fa_i16(_):
        ctx.call("qf_f_a_i16", _ffi.ptr(e16), B, _ffi.ptr(uo), _ffi.ptr(fl))

    def fa_packed(_):
        ctx.call("qf_f_a_packed", _ffi.ptr(pk), None, B, k, slot, _ffi.ptr(uo), _ffi.ptr(fl))

    fa_times = {"int16": [], "packed": []}
    for fn in (fa_i16, fa_packed, fa_i16, fa_packed):
        fn(0)
    for rnd in range(4):
        for fn, key in ((fa_i16, "int16"), (fa_packed, "packed")):
            fa_times[key].append(timed(fn, 0))
            assert np.array_equal(uo, u) and fl.all(), (name, key)
    rate = {key: B / float(np.median(v)) for key, v in times.items()}
    res.update({
        "samp_p_call_s": times, "samp_p_targets_per_s_median": rate,
        "packed_over_int16_rate": rate["packed"] / rate["int16"],
        "overflow_rows": overflow_rows, "nbytes_mean": float(np.mean(nb_mean)), "nbytes_max": nb_max,
        "nbytes_mean_expected": EXPECTED_MEAN[name], "packed_over_int16_bytes": float(np.mean(nb_mean)) / (2 * m),
        "d2h_bytes_per_call": {"int16": 2 * m * B, "packed": (slot + 4) * B},
        "f_a_call_s": fa_times,
        "f_a_targets_per_s_median": {key: B / float(np.median(v)) for key, v in fa_times.items()},
        "checked": {"rows_vs_samp_p": len(rows), "a_e_eq_u_rows": B},
    })
    # kernel times: one default chunk under the profiler, in a run of its own
    from torch.profiler import ProfilerActivity, profile

    C = min(B, 37888)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ctx.call("qf_samp_p_packed", _ffi.ptr(u), None, C, 5, 0, k, slot, _ffi.ptr(pk), _ffi.ptr(nb))
        ctx.call("qf_f_a_packed", _ffi.ptr(pk), None, C, k, slot, _ffi.ptr(uo), _ffi.ptr(fl))
        torch.cuda.synchronize()
    kern, total = {}, 0.0
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        total += t
        if "domain_encode_kernel" in ev.key or "domain_decode_kernel" in ev.key:
            kern["encode" if "encode" in ev.key else "decode"] = {"us": t, "calls": ev.count}
    res["profiled_chunk"] = {"targets": C, "kernels": kern, "all_kernels_us": total}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c2,c4")
    ap.add_argument("--calls", type=int, default=4)
    ap.add_argument("--check-rows", type=int, default=16)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_domain_code.json"))
    args = ap.parse_args()
    import torch

    import tools_b200 as T

    assert torch.cuda.is_available(), "needs a CUDA device"
    out = {"gpu": gpu_info(), "workloads": {}}
    for name in args.workloads.split(","):
        out["workloads"][name] = run_workload(T, name, args)
        print(name, json.dumps(out["workloads"][name]), flush=True)
    out["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"gpu": out["gpu"], "out": args.out}))


if __name__ == "__main__":
    main()
