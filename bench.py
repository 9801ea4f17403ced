#!/usr/bin/env python
"""bench.py -- samp_p preimages/s (+ f_a evals/s) of the B200 backend on the configurations BASELINE.json names.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c1|c2|c3|c4|c5] [--batch B] [--impl ours|reference]
                  [--dump-outputs DIR]

Default workload = BASELINE.json configs[1] (C2: PSFGPV n = 256, q = 2^24, 1M-target workload consumed in steps of
--batch targets per GPU); the default single-GPU run also carries `extra.rows`: C1, C3 (ring f_a / samp_p), C4 (one
PSFPerturbation shard, TrapGen's A_bar R timed separately) and C5 (compression, d in {1,4,10,11}), each with its own
roofline entry.  One JSON line on stdout (rank 0).  See DESIGN.md "Measurement" for what each key means."""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))


def gpv_s_for(n, m_bar):
    # SURVEY 8d: s = ceil((sqrt(m_bar)+1) * sqrt(5) * log2 n)   (bound from short_basis_classical.rs:233-235)
    return float(math.ceil((math.sqrt(m_bar) + 1.0) * math.sqrt(5.0) * math.log2(n)))


def gpv_s(gp):
    return gpv_s_for(gp.n, gp.m_bar)


def pert_s_for(m_bar, nk):
    # SURVEY 8d: s above sqrt(5 (s1(R)^2 + 1) + 1) with s1(R) ~ (sqrt(m_bar) + sqrt(nk)) / sqrt(2); 15 % margin
    s1 = (math.sqrt(m_bar) + math.sqrt(nk)) / math.sqrt(2)
    return float(math.ceil(1.15 * math.sqrt(5 * (s1 * s1 + 1) + 1)))


# name: kind, n, q, (r), default targets per step per GPU, description
WORKLOADS = {
    "c1": dict(kind="pert", n=8, q=64, r=3.0, s=25.0, batch=262144,
               desc="C1 README PSFPerturbation init_default(8, 64), r=3, s=25 (m=105), uniform synthetic targets"),
    "c2": dict(kind="gpv", n=256, q=2**24, batch=227328,  # six internal chunks of 2 x 148 SMs x 128 targets
               desc="C2 PSFGPV n=256 q=2^24 classical gadget (m=12352), uniform synthetic targets"),
    "c2small": dict(kind="gpv", n=64, q=2**24, batch=65536,
                    desc="reduced PSFGPV n=64 q=2^24 (m=3108) -- smoke-size variant, not the headline"),
    "c3": dict(kind="ring", n=256, q=3329, batch=131072,
               desc="C3 PSFGPVRing over X^256+1 mod 3329 (14 polynomials, D=3584), uniform synthetic targets"),
    "c4": dict(kind="pert", n=512, q=2**32 - 5, r=9.0, s=None, batch=60416,  # eight internal chunks of 7552 targets
               desc="C4 PSFPerturbation n=512 q=2^32-5 k=32 r=9 (m=32849), targets sharded over the GPUs"),
    "c5": dict(kind="compress", n=256, q=3329, batch=16 * 1024 * 1024,
               desc="C5 LossyCompressionFIPS203 compress/decompress on 16 Mi polynomials of degree 256 mod 3329"),
}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


DUMP_BYTES = 60_000_000  # --dump-outputs data budget: the .npy files stay under 64 MB with their headers


def dump_outputs(out_dir, rows_total, arrays):
    """--dump-outputs: write the same fixed, seeded sample of rows of every array as out_dir/<name>.npy.
    `arrays` maps a name to (device tensor whose first dimension is the row, numpy float dtype to store)."""
    import torch

    row_bytes = sum(t[0].numel() * np.dtype(dt).itemsize for t, dt in arrays.values())
    k = min(rows_total, DUMP_BYTES // row_bytes)
    rows = np.sort(np.random.default_rng(0).choice(rows_total, k, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, (t, dt) in arrays.items():
        x = t.index_select(0, torch.from_numpy(rows).to(t.device)).cpu().numpy()
        y = x.astype(dt)
        assert np.array_equal(y, x), f"{name}: values not exact in {np.dtype(dt).name}"
        np.save(os.path.join(out_dir, name + ".npy"), y)
    log(f"[dump] {k} of {rows_total} rows of {', '.join(arrays)} -> {out_dir}")


class ClockSampler:
    def __init__(self, gpu_index):
        self.cmd = ["nvidia-smi", f"--id={gpu_index}",
                    "--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                    "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                    "clocks_event_reasons.sw_power_cap", "--format=csv,noheader,nounits", "-lms", "200"]
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(self.cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ======================================================================================================================
# reference arm: the CPU restatement of the reference's own algorithm (oracle/) on the box's host threads
# ======================================================================================================================
def exact_abar_r(a_bar, r, q):
    """(A_bar R) mod q in float64 BLAS, exact: A_bar split into 12-bit limbs."""
    rf = r.astype(np.float64)
    acc = np.zeros((a_bar.shape[0], r.shape[1]), dtype=object)
    shift = 0
    rem = a_bar.astype(np.int64)
    while rem.any():
        limb = (rem & 0xFFF).astype(np.float64)
        part = np.rint(limb @ rf).astype(np.int64)
        acc = (acc + (part.astype(object) << shift)) % q
        rem >>= 12
        shift += 12
    return acc.astype(np.int64)


def oracle_classical_key(n, q, seed):
    """(A, R, gp) from the oracle's restatement of gen_trapdoor (gadget_classical.rs:56-68), numpy-vectorised product."""
    from oracle import qfall_oracle as O

    gp = O.GadgetParameters.init_default(n, q)
    rng = np.random.default_rng(seed)
    nk = n * gp.k
    a_bar = rng.integers(0, q, (n, gp.m_bar), dtype=np.int64)
    r = (rng.integers(0, 2, (gp.m_bar, nk)) - rng.integers(0, 2, (gp.m_bar, nk))).astype(np.int8)
    ar = exact_abar_r(a_bar, r, q)
    g = np.zeros((n, nk), dtype=np.int64)
    gvec = [pow(gp.base, t, q) for t in range(gp.k)]
    for j in range(n):
        g[j, j * gp.k:(j + 1) * gp.k] = gvec
    a = np.concatenate([a_bar, (g - ar) % q], axis=1)
    return gp, a, r


def oracle_short_basis(gp, a, r):
    """gen_short_basis_for_trapdoor (short_basis_classical.rs:54-110, tag = I) restated with numpy blocks:
    S = [[R S', I + R W],[S', W]], S' = I (x) S_k (columns reversed iff base^k = q), W = digits of -A[:, :m_bar]."""
    from oracle import qfall_oracle as O

    n, k, mb, q, base = gp.n, gp.k, gp.m_bar, gp.q, gp.base
    nk = n * k
    sk = np.array(O.short_basis_gadget_block(k, base, q), dtype=np.int64)
    sp = np.kron(np.eye(n, dtype=np.int64), sk)
    if base**k == q:
        sp = sp[:, ::-1]
    neg = (-a[:, :mb]) % q
    w = np.zeros((nk, mb), dtype=np.int64)
    for t in range(k):
        w[t::k, :] = (neg // base**t) % base
    rf = r.astype(np.float64)
    top_l = np.rint(rf @ sp.astype(np.float64)).astype(np.int64)
    top_r = np.eye(mb, dtype=np.int64) + np.rint(rf @ w.astype(np.float64)).astype(np.int64)
    return np.block([[top_l, top_r], [sp, w]])


def run_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from oracle import oracle_c as OC
    from oracle import qfall_oracle as O

    # torchrun exports OMP_NUM_THREADS=1; the (untimed) numpy key setup below would then run its BLAS calls on one
    # thread.  The timed part uses the C port's own pthreads (OC.threads()) and is not affected.
    try:
        from threadpoolctl import threadpool_limits

        threadpool_limits(limits=os.cpu_count() or 1)
    except Exception:
        pass
    import ctypes as C

    wl = WORKLOADS[args.workload]
    kind, n, q, desc = wl["kind"], wl["n"], wl["q"], wl["desc"]
    threads = OC.threads()
    rng = np.random.default_rng(2)
    lib = OC.lib()
    t0 = time.time()
    unit, metric = "preimages/s", "samp_p_preimages_per_s"
    if kind == "gpv":
        gp, a, r = oracle_classical_key(n, q, 2)
        s = gpv_s_for(n, gp.m_bar)
        basis = oracle_short_basis(gp, a, r)
        assert not ((a.astype(object) @ basis[:, :3].astype(object)) % q).any()  # basis columns lie in Lambda^perp(A)
        qr = np.linalg.qr(basis.astype(np.float64))
        gso = qr[0] * np.diag(qr[1])[None, :]
        piv, ainv = OC.unit_pivots(a[:, : 4 * n + 64], q)
        per_step = max(threads, args.ref_targets or threads)
        bt = np.ascontiguousarray(basis.astype(np.float64).T)
        gt = np.ascontiguousarray(gso.T)
        m = gp.m
        cfg = {"workload": desc, "targets_per_step": per_step, "s": s}
        sample = ("%d targets/step, one independent instance per thread; reference loop structure in fp64 (gpv.rs:152-161) "
                  "with the per-call Gaussian elimination hoisted out" % per_step)

        def step(seed):
            u = rng.integers(0, q, (per_step, n), dtype=np.int64)
            e = np.empty((per_step, m), dtype=np.int32)
            lib.orc_samp_p_gpv(C.c_void_p(bt.ctypes.data), C.c_void_p(gt.ctypes.data), C.c_void_p(piv.ctypes.data),
                               C.c_void_p(ainv.ctypes.data), C.c_long(len(piv)), C.c_void_p(u.ctypes.data),
                               C.c_void_p(e.ctypes.data), C.c_long(per_step), C.c_long(n), C.c_long(m), C.c_uint64(q),
                               C.c_double(s), C.c_uint64(seed), C.c_int(threads))
            return u, e, per_step

        def verify(u, e):
            assert np.array_equal(O.f_a_classical_batch(a, e[:2], q), u[:2])
    elif kind == "pert":
        gp, a, r = oracle_classical_key(n, q, 2)
        rr = wl["r"]
        s = wl["s"] or pert_s_for(gp.m_bar, n * gp.k)
        lmat = O.compute_sqrt_sigma_2(r, s, rr, 2)
        sb = np.array(O.short_basis_gadget(gp), dtype=np.float64)
        sg = O.gso_f64(sb)
        per_step = max(threads, args.ref_targets or (threads * (64 if gp.m < 1000 else 1)))
        cfg = {"workload": desc, "targets_per_step": per_step, "s": s, "r": rr}
        sample = ("%d targets/step, one independent instance per thread; reference loop structure in fp64 "
                  "(mp_perturbation.rs:304-336: dense sqrt(Sigma_2) product, dense nk x nk gadget nearest plane)" % per_step)

        def step(seed):
            u = rng.integers(0, q, (per_step, n), dtype=np.int64)
            e = OC.samp_p_pert(lmat, a, r, sb, sg, u, n, gp.k, gp.m_bar, 2, q, rr, seed, threads)
            return u, e, per_step

        def verify(u, e):
            assert np.array_equal(O.f_a_classical_batch(a, e[:2], q), u[:2])
    elif kind == "ring":
        gp = O.GadgetParametersRing.init_default(n, q)
        s = ((2 * 2 * 1.005 * math.sqrt(n) + 1) * 2) * 4
        a_bar = [int(x) for x in rng.integers(0, q, n)]
        rt = [[int(x) for x in np.rint(rng.normal(0, 1.005 / math.sqrt(2 * math.pi), n))] for _ in range(gp.k)]
        et = [[int(x) for x in np.rint(rng.normal(0, 1.005 / math.sqrt(2 * math.pi), n))] for _ in range(gp.k)]
        a = O.gen_trapdoor_ring_lwe(gp, a_bar, rt, et)
        emb = np.array(O.coeff_embed(O.gen_short_basis_for_trapdoor_ring(gp, a, rt, et), n), dtype=np.float64)
        gso = O.gso_f64(emb)
        piv = np.arange(n, dtype=np.int32)
        ainv = np.eye(n, dtype=np.int64)
        per_step = max(threads, args.ref_targets or threads * 8)
        bt, gt = np.ascontiguousarray(emb.T), np.ascontiguousarray(gso.T)
        d = emb.shape[0]
        cfg = {"workload": desc, "targets_per_step": per_step, "s": s}
        sample = ("%d targets/step; GPV08 SampleD on the embedded basis in fp64 with the basis and its GSO built ONCE "
                  "(the reference rebuilds both per call, gpv_ring.rs:169,205-211 -- favours the CPU arm)" % per_step)

        def step(seed):
            u = rng.integers(0, q, (per_step, n), dtype=np.int64)
            e = np.empty((per_step, d), dtype=np.int32)
            lib.orc_samp_p_gpv(C.c_void_p(bt.ctypes.data), C.c_void_p(gt.ctypes.data), C.c_void_p(piv.ctypes.data),
                               C.c_void_p(ainv.ctypes.data), C.c_long(n), C.c_void_p(u.ctypes.data), C.c_void_p(e.ctypes.data),
                               C.c_long(per_step), C.c_long(n), C.c_long(d), C.c_uint64(q), C.c_double(s), C.c_uint64(seed),
                               C.c_int(threads))
            return u, e, per_step

        def verify(u, e):
            assert O.f_a_ring(a, e[0].reshape(gp.k + 2, n).tolist(), n, q) == u[0].tolist()
    else:  # compress
        unit, metric = "GB/s", "lossy_compress_GBps"
        count = (args.ref_targets or 2 * 1024 * 1024) * 256
        x = rng.integers(0, q, count).astype(np.uint16)
        cfg = {"workload": desc, "polys_per_step": count // 256, "d": 10}
        sample = "%d polynomials/step, d = 10, all host threads (lossy_compression_fips203.rs:101-111 per coefficient)" % (count // 256)

        def step(seed):
            y = OC.compress_u16(x, q, 10, False, threads)
            return x, y, count * 4 / 1e9

        def verify(u, e):
            assert np.array_equal(e[:1000].astype(np.uint64), O.lossy_compress_np(u[:1000], 10, q))
    log(f"[reference] key setup {time.time() - t0:.1f}s (untimed)")
    for w in range(args.warmup):
        step(w)
    t0 = time.perf_counter()
    units = 0
    for k in range(args.steps):
        u, e, cnt = step(100 + k)
        units += cnt
    dt = time.perf_counter() - t0
    verify(u, e)
    val = units / dt
    line = {
        "impl": "reference", "metric": metric, "value": val, "unit": unit,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64" if kind != "compress" else "u16",
        "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": val, "unit": unit, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ======================================================================================================================
# our arm
# ======================================================================================================================
def measure_i8_peak(local):
    """Measured int8 tensor-pipe ceiling (qf_probe_i8_peak): burst and sustained TOP/s of a plain one-digit-pair
    tcgen05 kind::i8 contraction with long K."""
    from tools_b200 import _ffi

    best, sus, pipe = _ffi.C.c_double(), _ffi.C.c_double(), _ffi.C.c_double()
    st = _ffi.lib().qf_probe_i8_peak(local, 37888, 8192, 16384, 8, 1500.0, _ffi.C.byref(best), _ffi.C.byref(sus),
                                     _ffi.C.byref(pipe))
    if st != 0 or best.value <= 0:
        return None
    return {"pipe_tops": pipe.value, "gemm_burst_tops": best.value, "gemm_sustained_tops": sus.value,
            "how": "qf_probe_i8_peak.  pipe: every SM repeats the tcgen05.mma kind::i8 instructions of one shared-memory-resident "
                   "128 x 256 x 128 block (no operand traffic: 100 % pipe activity), best of 3.  gemm: 37888 x 8192 x 16384 u8 x s8 "
                   "contraction (LX = LW = 1, 128 x 256 tiles, cta_group::1, double-buffered TMEM, int32 store) on random bytes, "
                   "best of 8 launches (burst) and back to back for 1.5 s (sustained): bound by the L2 -> shared-memory operand "
                   "feed of a one-CTA tiling, not by the pipe"}


def compress_headline(args, torch, dev, rank, world, local, barrier):
    """--workload c5: compress + decompress GB/s at d = 10 over all ranks (shard by polynomial index, no collective)."""
    import bench_rows as BR
    from tools_b200.compression import compress_dev

    npoly = args.batch or WORKLOADS["c5"]["batch"]
    count = npoly * 256
    gen = torch.Generator(device=dev)
    gen.manual_seed(1000 + rank)  # the same inputs on every run, distinct per rank
    x = torch.randint(0, 3329, (count,), dtype=torch.int32, device=dev, generator=gen).to(torch.int16)
    y = torch.empty_like(x)
    st = torch.cuda.current_stream().cuda_stream
    for _ in range(args.warmup):
        compress_dev(x.data_ptr(), y.data_ptr(), count, 3329, 10, st)
    clocks = ClockSampler(local)
    barrier()
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        compress_dev(x.data_ptr(), y.data_ptr(), count, 3329, 10, st)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    clock_info = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, npoly, {"compress_in": (x.view(npoly, 256), np.float32),
                                                "compress_out": (y.view(npoly, 256), np.float32)})
    if world > 1:
        import torch.distributed as dist

        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = world * args.steps * count * 4 / (ms * 1e-3) / 1e9
    # end to end: pinned host buffers through qf_compress_u16 (H2D + D2H inside)
    from tools_b200 import _ffi

    e2e_count = 1 << 28
    hx = torch.empty(e2e_count, dtype=torch.int16).pin_memory()
    hy = torch.empty(e2e_count, dtype=torch.int16).pin_memory()
    hx.copy_(x[:e2e_count].cpu())
    lib = _ffi.lib()
    lib.qf_compress_u16(_ffi.ptr(hx.numpy()), _ffi.ptr(hy.numpy()), e2e_count, 3329, 10, 0, None)
    t0 = time.perf_counter()
    for _ in range(3):
        assert lib.qf_compress_u16(_ffi.ptr(hx.numpy()), _ffi.ptr(hy.numpy()), e2e_count, 3329, 10, 0, None) == 0
    e2e_dt = (time.perf_counter() - t0) / 3
    if rank != 0:
        return
    rows = BR.row_compress(dev, npoly) if world == 1 else []
    line = {"metric": "lossy_compress_GBps", "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u16", "data": "synthetic",
            "config": {"workload": WORKLOADS["c5"]["desc"], "polys_per_step_per_gpu": npoly, "d": 10,
                       "l2": "17 GB per pass, far beyond L2"},
            "e2e": {"value": world * e2e_count * 4 / e2e_dt / 1e9, "unit": "GB/s", "h2d_bytes_per_step": e2e_count * 2,
                    "d2h_bytes_per_step": e2e_count * 2},
            "gpu_launches": args.steps,
            "roofline": BR.hbm_roofline("compress_u16_kernel", count * 4, ms / args.steps, "compress_u16_kernel"),
            "cpu_baseline": None, "clocks": clock_info, "extra": {"rows": rows}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=0, help="targets per step per GPU (0 = workload default)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--ref-targets", type=int, default=0, help="reference arm: targets per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra.rows block of the default run")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a fixed, seeded sample (<= 64 MB) of the last timed step's results to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of --impl ours")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)

    import torch

    import tools_b200 as T
    from tools_b200 import _ffi

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    wl = WORKLOADS[args.workload]
    kind, n, q, desc = wl["kind"], wl["n"], wl["q"], wl["desc"]
    if kind == "compress":
        compress_headline(args, torch, dev, rank, world, local, barrier)
        if world > 1:
            dist.destroy_process_group()
        return
    batch = args.batch or wl["batch"]
    t0 = time.time()
    r_par = 1.0
    if kind == "gpv":
        gp = T.GadgetParameters.init_default(n, q)
        s = gpv_s(gp)
        psf = T.PSFGPV(gp, s, device=local)
        dim, dom_shape = gp.m, (gp.m,)
    elif kind == "pert":
        gp = T.GadgetParameters.init_default(n, q)
        r_par = wl["r"]
        s = wl["s"] or pert_s_for(gp.m_bar, n * gp.k)
        psf = T.PSFPerturbation(gp, r_par, s, device=local)
        dim, dom_shape = gp.m, (gp.m,)
    else:
        gp = T.GadgetParametersRing.init_default(n, q)
        s = ((2 * 2 * 1.005 * math.sqrt(n) + 1) * 2) * 4  # gpv_ring.rs:296-298
        psf = T.PSFGPVRing(gp, s, 1.005, device=local)
        dim, dom_shape = n * (gp.k + 2), (gp.k + 2, n)
    ctx = psf.ctx
    if kind != "ring":
        psf.trap_gen(seed=1)  # untimed: the first launch of a kernel loads its module (tens of ms), not TrapGen's work
    ctx.call("qf_profile", 1)
    t0 = time.time()
    a, td = psf.trap_gen(seed=2)  # same seed on every rank: the key is replicated, not communicated
    t_trapgen = time.time() - t0
    tg = [_ffi.C.c_double() for _ in range(6)]
    tgl = [_ffi.C.c_uint64() for _ in range(2)]
    ctx.call("qf_profile_read", _ffi.C.byref(tg[0]), _ffi.C.byref(tg[1]), _ffi.C.byref(tgl[0]), _ffi.C.byref(tg[2]),
             _ffi.C.byref(tg[3]), _ffi.C.byref(tg[4]), _ffi.C.byref(tgl[1]))
    ctx.call("qf_profile", 0)
    trapgen_info = {"trap_gen_s": t_trapgen,
                    "abar_r_tcgen05": {"ms": tg[2].value, "useful_ops": tg[3].value,
                                       "TOPs": tg[3].value / tg[2].value / 1e9 if tg[2].value else None,
                                       "launches": int(tgl[1].value)} if kind != "ring" else None}
    psf._install_a(a)
    psf._install_td(a, td)
    log(f"[rank {rank}] key setup {time.time() - t0:.1f}s  dim={dim} s={s} batch/step/gpu={batch}")
    # a dedicated (non-default) stream shared by torch's events and the library's launches
    tstream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0
    ctx.call("qf_set_stream", _ffi.ptr(stream))
    lib = _ffi.lib()

    total_steps = args.warmup + args.steps
    u = torch.empty((batch, n), dtype=torch.int64, device=dev)
    e = torch.empty((batch,) + dom_shape, dtype=torch.int32, device=dev)

    def fill_targets(step_idx):
        # Philox-seeded uniform targets, distinct per (rank, step)
        st = lib.qf_fill_uniform_modq_dev(_ffi.ptr(u.data_ptr()), u.numel(), q, 1000 + rank * 100003 + step_idx,
                                          _ffi.ptr(stream))
        assert st == 0

    def step(step_idx):
        first = (rank * total_steps + step_idx) * batch
        ctx.call("qf_samp_p_dev", _ffi.ptr(u.data_ptr()), batch, 2, first, _ffi.ptr(e.data_ptr()))

    # ---- device-resident throughput ------------------------------------------------------------------
    for w in range(args.warmup):
        fill_targets(w)
        step(w)
    ctx.call("qf_synchronize")
    fill_targets(args.warmup)
    clocks = ClockSampler(local)
    barrier()
    if rank == 0:
        clocks.start()
    ctx.call("qf_profile", 1)
    l0 = ctx.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for k in range(args.steps):
        step(args.warmup + k)
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    launches = ctx.launch_count() - l0
    gms, gfl, gln = _ffi.C.c_double(), _ffi.C.c_double(), _ffi.C.c_uint64()
    ims, iops, iiss, iln = _ffi.C.c_double(), _ffi.C.c_double(), _ffi.C.c_double(), _ffi.C.c_uint64()
    ctx.call("qf_profile_read", _ffi.C.byref(gms), _ffi.C.byref(gfl), _ffi.C.byref(gln), _ffi.C.byref(ims),
             _ffi.C.byref(iops), _ffi.C.byref(iiss), _ffi.C.byref(iln))
    ctx.call("qf_profile", 0)
    clock_info = clocks.stop() if rank == 0 else None
    ctx.call("qf_synchronize")
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = world * args.steps * batch / (ms * 1e-3)

    # correctness of what was just timed: A e = u for the last step (oracle-free, through f_a_dev)
    uo = torch.empty_like(u)
    fl = torch.empty(batch, dtype=torch.uint8, device=dev)
    ctx.call("qf_f_a_dev", _ffi.ptr(e.data_ptr()), batch, _ffi.ptr(uo.data_ptr()), _ffi.ptr(fl.data_ptr()))
    ctx.call("qf_synchronize")
    assert torch.equal(uo, u), "A e != u in the timed output"
    assert bool(fl.all()), "a timed preimage fails check_domain"
    # spherical law: E||e||^2 = dim (s r)^2 / (2 pi) for D_{Lambda_u^perp(A), s r}
    norm_ratio = float((e[:4096].double() ** 2).reshape(min(batch, 4096), -1).sum(1).mean().item()
                       / (dim * (s * r_par) ** 2 / (2 * math.pi)))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, batch, {"samp_p_e": (e, np.float32), "samp_p_u": (u, np.float64)})

    # ---- f_a evals/s (device resident; sigma = the preimages, in domain) ---------------------------------
    for _ in range(3):
        ctx.call("qf_f_a_dev", _ffi.ptr(e.data_ptr()), batch, _ffi.ptr(uo.data_ptr()), _ffi.ptr(fl.data_ptr()))
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    fa_steps = max(args.steps, 4)
    for _ in range(fa_steps):
        ctx.call("qf_f_a_dev", _ffi.ptr(e.data_ptr()), batch, _ffi.ptr(uo.data_ptr()), _ffi.ptr(fl.data_ptr()))
    f1.record()
    barrier()
    fa_ms = f0.elapsed_time(f1)
    if world > 1:
        t = torch.tensor([fa_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        fa_ms = float(t.item())
    fa_value = world * fa_steps * batch / (fa_ms * 1e-3)

    # ---- final gather over NVLink (SURVEY K12 / 8e): the last step's shards, narrowed to int16 on the device, are
    # gathered to rank 0 with one NCCL gather when they fit there; verified on rank 0 against the gathered targets --------
    gather_info = None
    if world > 1:
        from tools_b200.sharding import gather_domain_i16

        gather_info = gather_domain_i16(torch, dist, lib, _ffi, e, u, rank, world, dev, tstream, max_bytes=64 << 30)
        if rank == 0 and gather_info and gather_info.get("gathered") is not None:
            ge, gu = gather_info.pop("gathered")
            # rank 0 checks the LAST rank's shard with its own (replicated) key: A e = u
            lo = (world - 1) * batch
            chk_e = ge[lo:lo + min(batch, 8192)].to(torch.int32).contiguous()
            chk_u = torch.empty((chk_e.shape[0], n), dtype=torch.int64, device=dev)
            chk_f = torch.empty(chk_e.shape[0], dtype=torch.uint8, device=dev)
            ctx.call("qf_f_a_dev", _ffi.ptr(chk_e.data_ptr()), chk_e.shape[0], _ffi.ptr(chk_u.data_ptr()), _ffi.ptr(chk_f.data_ptr()))
            ctx.call("qf_synchronize")
            assert torch.equal(chk_u, gu[lo:lo + chk_e.shape[0]]) and bool(chk_f.all()), "gathered shard: A e != u"
            gather_info["verified"] = "A e = u on the last rank's gathered shard (rank 0, replicated key)"
            del ge, gu, chk_e, chk_u, chk_f
        elif gather_info:
            gather_info.pop("gathered", None)

    # ---- end to end through the host-buffer C ABI (pinned host memory, H2D + D2H inside) ----------------
    # int16 Domain form when every entry fits (|e_i| <= 6 s r < 2^15: C2, C3; not C1/C4 sized s r), else int32
    e2e_i16 = 6.5 * s * r_par < 32767
    # host result buffer (pinned) of at most 8 GiB; otherwise a whole number of 1024-target blocks that fits
    e2e_esz = 2 if e2e_i16 else 4
    e2e_batch = batch if dim * batch * e2e_esz <= (8 << 30) else max(1024, ((8 << 30) // (dim * e2e_esz)) // 1024 * 1024)
    hu = torch.empty((e2e_batch, n), dtype=torch.int64).pin_memory()
    he = torch.empty((e2e_batch,) + dom_shape, dtype=torch.int16 if e2e_i16 else torch.int32).pin_memory()
    hu.copy_(u[:e2e_batch].cpu())
    hu_np, he_np = hu.numpy(), he.numpy()
    e2e_fn = "qf_samp_p_i16" if e2e_i16 else "qf_samp_p"

    def e2e_step(i):
        ctx.call(e2e_fn, _ffi.ptr(hu_np), e2e_batch, 2, (rank * 1000 + i) * e2e_batch, _ffi.ptr(he_np))

    e2e_step(0)
    barrier()
    t0 = time.perf_counter()
    e2e_steps = max(2, min(args.steps, 4))
    for i in range(e2e_steps):
        e2e_step(1 + i)
    torch.cuda.synchronize()
    e2e_dt = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_dt], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_dt = float(t.item())
    e2e_value = world * e2e_steps * e2e_batch / e2e_dt
    if kind != "ring":
        assert np.array_equal(he_np[:4].astype(np.int64) @ a.T % q, hu_np[:4])

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernels -----------------------------------------------------------------------
    import bench_rows as BR

    peaks = BR.PEAKS
    # fp64: MEASURED_PEAKS.json has no fp64 entry: measure the cuBLAS DGEMM burst the same way the driver measured
    # bf16 (torch.matmul 8192^3, best of 6) and use it as the denominator.
    x = torch.randn(8192, 8192, dtype=torch.float64, device=dev)
    y = torch.randn(8192, 8192, dtype=torch.float64, device=dev)
    best = 1e9
    for _ in range(6):
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        torch.matmul(x, y)
        p1.record()
        torch.cuda.synchronize()
        best = min(best, p0.elapsed_time(p1))
    dgemm_tf = 2 * 8192**3 / (best * 1e-3) / 1e12
    del x, y
    i8 = measure_i8_peak(local)
    bf16 = peaks.get("bf16_tflops")
    if i8:
        # denominator = the measured ceiling of the pipe itself (the most demanding of the measured figures)
        i8_peak = max(i8["pipe_tops"], i8["gemm_burst_tops"])
        i8_src = "measured in this run (pipe_tops): " + i8["how"]
    else:
        i8_peak = 2.0 * (bf16 or 1590.0)
        i8_src = "2 x the bf16 burst (probe failed)"
    f64_achieved = gfl.value / (gms.value * 1e-3) / 1e12 if gms.value > 0 else None
    f64_roof = {
        "kernel": "gemm_f64_kernel (mma.sync.m8n8k4.f64 DMMA): nearest-plane updates inside 1024-blocks, centre -> GSO map",
        "bound": "tensor", "achieved": f64_achieved, "peak": dgemm_tf, "unit": "TFLOP/s",
        "frac": (f64_achieved / dgemm_tf) if f64_achieved else None, "traffic": None,
        "peak_source": "cuBLAS DGEMM 8192^3 burst measured in this run (MEASURED_PEAKS.json has no fp64 entry; nominal ~37 TF/s)",
        "kernel_ms_per_step": gms.value / args.steps, "kernel_share_of_step": gms.value / ms, "launches": int(gln.value),
    }
    if ims.value > 0:
        issued = iiss.value / (ims.value * 1e-3) / 1e12
        algo = iops.value / (ims.value * 1e-3) / 1e12
        tr = BR.profile_traffic("gemm_i8_kernel") or {}
        # dominant kernel of the step.  `achieved` counts the ALGORITHMIC contraction 2*B*N*K of every launch
        # (the exact integer / fixed-point product the reference computes in big-number arithmetic); the tensor pipe
        # executes that once per digit pair (`issued`).
        roofline = {
            "kernel": "gemm_i8_kernel (tcgen05.mma kind::i8, TMA, TMEM): fixed-point nearest-plane updates U*z, centre maps "
                      "(Mt_1 z2, M' g3) and exact integer products (A_bar z2, R e_bot; S z in the one-pass form)" if kind != "pert" else
                      "gemm_i8_kernel (tcgen05.mma kind::i8, TMA, TMEM): x2 = sqrt(Sigma_2) g (fixed point), v = u - A p, e = p + [R;I] z",
            "bound": "tensor", "achieved": algo, "peak": i8_peak, "unit": "TOP/s", "frac": algo / i8_peak,
            "achieved_issued": issued, "frac_issued": issued / i8_peak,
            "algorithmic_ops": "2*B*N*K per launch (B targets x N coordinates x K contraction length), summed over the "
                               "launches of the timed region; `issued` multiplies by the digit pairs the tensor pipe "
                               "actually executed (zero digit planes skipped), counted by the kernel",
            "traffic": tr.get("dram_bytes"), "traffic_note": tr.get("note"),
            "peak_source": i8_src, "i8_peak_probe": i8, "digit_pairs_per_mac": issued / algo if algo else None,
            "kernel_ms_per_step": ims.value / args.steps, "kernel_share_of_step": ims.value / ms, "launches": int(iln.value),
        }
    else:
        roofline = f64_roof

    # ---- CPU baseline: the oracle's C restatement on a bounded sample ----------------------------------
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            cpu = cpu_baseline(kind, psf, gp, a, td, hu_np, n, q, s, r_par)
        except Exception as ex:  # the baseline is reported, never required
            cpu = {"value": None, "error": repr(ex)}

    line = {
        "metric": "samp_p_preimages_per_s", "value": value, "unit": "preimages/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": desc, "targets_per_step_per_gpu": batch, "total_targets_timed": world * args.steps * batch,
                   "note": "the configuration's target count is consumed in steps of targets_per_step_per_gpu (HBM workspace); "
                           "throughput does not depend on the number of steps",
                   "s": s, "r": r_par if kind == "pert" else None,
                   "l2": "per-step working set (T, Z: batch x dim fp64 = %.1f GB each) exceeds L2" % (batch * dim * 8 / 1e9),
                   "sharding": "targets split across ranks, key replicated, no collective on the data path"},
        "e2e": {"value": e2e_value, "unit": "preimages/s", "h2d_bytes_per_step": e2e_batch * n * 8,
                "d2h_bytes_per_step": e2e_batch * dim * (2 if e2e_i16 else 4), "steps": e2e_steps,
                "targets_per_step_per_gpu": e2e_batch, "domain_dtype": "int16" if e2e_i16 else "int32", "entry": e2e_fn},
        "f_a": {"value": fa_value, "unit": "evals/s", "ms_per_step": fa_ms / fa_steps},
        "gpu_launches": int(launches),
        "checks": {"A_e_equals_u_all_targets_last_step": True, "check_domain_all": True,
                   "mean_norm2_over_dim_s2_2pi": norm_ratio},
        "roofline": roofline,
        "roofline_f64": f64_roof,
        "key_setup": trapgen_info,
        "gather": gather_info,
        "cpu_baseline": cpu,
        "clocks": clock_info,
    }
    # ---- the other configurations of BASELINE.json, device resident, each with its own roofline ----------------
    if world == 1 and args.workload == "c2" and not args.no_extra:
        del u, e, uo, fl, hu, he
        psf.ctx.close()
        torch.cuda.set_stream(torch.cuda.default_stream(dev))
        torch.cuda.empty_cache()
        rows = []
        plan = [("compress", lambda: BR.row_compress(dev)), ("encode", lambda: BR.row_encode(dev, ds=(10,))),
                ("ring", lambda: BR.row_ring(dev)),
                ("pert_c4", lambda: [BR.row_pert(dev, *BR.c4_params(), 15104,
                                                 "C4 PSFPerturbation n=512 q=2^32-5 k=32 r=9 (one GPU shard)", i8_peak=i8_peak)]),
                ("pert_c1", lambda: [BR.row_pert(dev, 8, 64, 3.0, 25.0, 262144, "C1 README PSFPerturbation n=8 q=64 r=3 s=25",
                                                 i8_peak=i8_peak)])]
        for name, fn in plan:
            try:
                rows.extend(fn())
            except Exception as ex:
                rows.append({"row": name, "error": repr(ex)})
            torch.cuda.empty_cache()
        line["extra"] = {"rows": rows}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def cpu_baseline(kind, psf, gp, a, td, hu_np, n, q, s, r_par):
    """The oracle's C restatement of the reference loop on a bounded sample of the same workload (rank 0, N = 1)."""
    import ctypes as C

    from oracle import oracle_c as OC

    threads = OC.threads()
    if kind == "gpv":
        sample = threads  # one target per thread: ~ one pass over the 2.4 GB of basis + GSO each
        sb, sg = td
        if sg is None:  # the backend kept the GSO on the device: fetch a host copy for the CPU arm (untimed)
            sg = psf.gso(sb)
        t1 = time.perf_counter()
        piv, ainv = OC.unit_pivots(a[:, : 4 * n + 64], q)
        us = np.ascontiguousarray(hu_np[:sample])
        bt = np.ascontiguousarray(np.asarray(sb, dtype=np.float64).T)  # rows = basis vectors (untimed layout change)
        gt = np.ascontiguousarray(np.asarray(sg, dtype=np.float64).T)
        ec = np.empty((sample, gp.m), dtype=np.int32)
        tc = time.perf_counter()
        OC.lib().orc_samp_p_gpv(C.c_void_p(bt.ctypes.data), C.c_void_p(gt.ctypes.data), C.c_void_p(piv.ctypes.data),
                                C.c_void_p(ainv.ctypes.data), C.c_long(len(piv)), C.c_void_p(us.ctypes.data),
                                C.c_void_p(ec.ctypes.data), C.c_long(sample), C.c_long(n), C.c_long(gp.m), C.c_uint64(q),
                                C.c_double(s), C.c_uint64(1), C.c_int(threads))
        dtc = time.perf_counter() - tc
        assert np.array_equal(ec[:2].astype(np.int64) @ a.T % q, us[:2])
        return {"value": sample / dtc, "unit": "preimages/s", "cores": threads, "kind": "port",
                "sample": f"{sample} targets of the same workload, one per host thread ({dtc:.1f}s); reference "
                          "loop structure in fp64 with the per-call Gaussian elimination hoisted out "
                          f"(setup {tc - t1:.1f}s untimed)"}
    if kind == "pert":
        rmat, l, (sb, sg) = td
        if gp.m > 4096:
            return {"value": None, "unit": "preimages/s", "cores": threads, "kind": "port",
                    "sample": "not run in the default bench: the dense m x m sqrt(Sigma_2) and nk x nk gadget GSO the reference "
                              "loop needs are 8.6 + 4.3 GB of host doubles at C4 (`bench.py --impl reference --workload c4` runs it)"}
        if l is None:
            l = psf.compute_sqrt_sigma_2(rmat)
        from oracle import qfall_oracle as O

        sbf = np.array(O.short_basis_gadget(O.GadgetParameters.init_default(n, q)), dtype=np.float64)
        sample = threads * 256
        us = np.ascontiguousarray(hu_np[:sample])
        tc = time.perf_counter()
        ec = OC.samp_p_pert(l, a, rmat, sbf, O.gso_f64(sbf), us, n, gp.k, gp.m_bar, 2, q, r_par, 1, threads)
        dtc = time.perf_counter() - tc
        assert np.array_equal(ec[:2].astype(np.int64) @ a.T % q, us[:2])
        return {"value": sample / dtc, "unit": "preimages/s", "cores": threads, "kind": "port",
                "sample": f"{sample} targets, reference loop structure in fp64 (mp_perturbation.rs:304-336), {dtc:.2f}s"}
    return {"value": None, "unit": "preimages/s", "cores": threads, "kind": "port",
            "sample": "ring: `bench.py --impl reference --workload c3`"}


if __name__ == "__main__":
    main()
