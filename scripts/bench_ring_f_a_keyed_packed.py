"""Keyed ring f_a on packed sigma (qf_ring_f_a_keyed_packed[_dev], DESIGN.md 4.13) against the int32 keyed calls at C3
(X^256 + 1, q = 3329, k = 12: 14 polynomials, D = 3584, s = 522.6).

sigma comes from qf_samp_d_dev; the slots are its code at the parameters of qf_domain_code_params.  262 144 signatures per
pass (3.8 GB as int32, about 1.2 GB packed: both far larger than the 126 MB L2).  Key tables of T = 1, 4096 and 65 536
uniform keys, key indices in random order.  Every variant alternates with the others in each of two rounds:
  device-resident (CUDA events around one call over the batch; 2 warm-up passes, then about half a second of passes):
    dev_int32     qf_ring_f_a_keyed_dev on the int32 rows;
    dev_compose   qf_domain_decode_dev into an int32 buffer, qf_ring_f_a_keyed_dev on it, and the AND of the two flags;
    dev_fused     qf_ring_f_a_keyed_packed_dev;
  host-fed, from pinned host buffers (host clock around the synchronous call, the same pass count rule):
    host_int32    qf_ring_f_a_keyed;
    host_packed   qf_ring_f_a_keyed_packed.
Every timed output is checked against qf_ring_f_a_keyed_dev on the int32 rows: every row for the device variants, 64 seeded
rows for the host ones.  Writes one JSON file with the card name and power limit.

  python scripts/bench_ring_f_a_keyed_packed.py [--out FILE] [--quick]
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
KEY_COUNTS = (1, 4096, 65536)
SAMPLE = 64


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in out.split(",")]
    return {"name": name, "power_limit": power}


def timed_dev(torch, fn, min_s):
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


def timed_host(fn, min_s):
    fn()
    t0 = time.perf_counter()
    fn()
    one = time.perf_counter() - t0
    reps = max(1, min(1000, int(math.ceil(min_s / max(one, 1e-6)))))
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    return (time.perf_counter() - t0) / reps


T0 = time.perf_counter()


def log(msg):
    print(f"[{time.perf_counter() - T0:7.1f} s] {msg}", flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_ring_f_a_keyed_packed.json"))
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
    psf = T.PSFGPVRing(gp, s, 1.005)
    kc, slot = psf.domain_code_params()
    res = {"gpu": gpu_info(), "workload": f"C3 ring f_a with a key per target, n = {N}, q = {Q}, k = {gp.k}, D = {d}, "
                                          f"s = {s:.1f}, {B} signatures per pass, key indices in random order", "batch": B}
    stream = torch.cuda.current_stream(dev).cuda_stream  # the library runs where the CUDA events are recorded
    psf.ctx.call("qf_set_stream", _ffi.ptr(stream))
    lib = _ffi.lib()

    sig = torch.empty((B, d), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    psf.ctx.call("qf_samp_d_dev", B, 5, 0, _ffi.ptr(sig.data_ptr()))
    psf.ctx.call("qf_synchronize")
    from tools_b200 import domain_code

    packed, nbytes = domain_code.encode(sig, kc, slot)
    torch.cuda.synchronize()
    assert bool((nbytes > 0).all())
    res["code"] = {"k": kc, "slot_bytes": slot, "mean_nbytes": float(nbytes.double().mean()), "max_nbytes": int(nbytes.max()),
                   "int32_bytes": d * 4, "h2d_bytes_per_signature_int32": d * 4 + 4,
                   "h2d_bytes_per_signature_packed": slot + 4}
    log(f"sigma and slots ready: k = {kc}, slot {slot} bytes, mean code {res['code']['mean_nbytes']:.0f} bytes")
    stage = torch.empty((B, d), dtype=torch.int32, device=dev)  # the int32 rows of dev_compose
    ok_c = torch.empty(B, dtype=torch.uint8, device=dev)
    u = torch.empty((B, N), dtype=torch.int64, device=dev)
    fl = torch.empty(B, dtype=torch.uint8, device=dev)
    u_ref = torch.empty((B, N), dtype=torch.int64, device=dev)
    fl_ref = torch.empty(B, dtype=torch.uint8, device=dev)
    sig_h = torch.empty((B, d), dtype=torch.int32).pin_memory()
    sig_h.copy_(sig.cpu())
    packed_h = torch.empty((B, slot), dtype=torch.uint8).pin_memory()
    packed_h.copy_(packed.cpu())
    u_h = torch.empty((B, N), dtype=torch.int64).pin_memory()
    fl_h = torch.empty(B, dtype=torch.uint8).pin_memory()
    sample = torch.from_numpy(rng.choice(B, SAMPLE, replace=False))
    log("host buffers pinned")

    tables = {}
    for t in KEY_COUNTS:
        idx = rng.integers(0, t, B).astype(np.int32)
        tables[t] = dict(keys=np.ascontiguousarray(rng.integers(0, Q, (t, gp.k + 2, N), dtype=np.int64)),
                         idx=torch.from_numpy(idx).to(dev), idx_h=torch.from_numpy(idx).pin_memory())

    P = _ffi.ptr

    def dev_int32(ix):
        return lambda: psf.ctx.call("qf_ring_f_a_keyed_dev", P(sig.data_ptr()), P(ix.data_ptr()), B, P(u.data_ptr()),
                                    P(fl.data_ptr()))

    def dev_compose(ix):
        def run():
            st = lib.qf_domain_decode_dev(P(packed.data_ptr()), B, d, kc, slot, P(stage.data_ptr()), P(ok_c.data_ptr()),
                                          P(stream))
            assert st == _ffi.QF_OK
            psf.ctx.call("qf_ring_f_a_keyed_dev", P(stage.data_ptr()), P(ix.data_ptr()), B, P(u.data_ptr()), P(fl.data_ptr()))
            fl.mul_(ok_c)
        return run

    def dev_fused(ix):
        return lambda: psf.ctx.call("qf_ring_f_a_keyed_packed_dev", P(packed.data_ptr()), P(ix.data_ptr()), B, kc, slot,
                                    P(u.data_ptr()), P(fl.data_ptr()))

    def host_int32(ixh):
        return lambda: psf.ctx.call("qf_ring_f_a_keyed", P(sig_h.data_ptr()), P(ixh.data_ptr()), B, P(u_h.data_ptr()),
                                    P(fl_h.data_ptr()))

    def host_packed(ixh):
        return lambda: psf.ctx.call("qf_ring_f_a_keyed_packed", P(packed_h.data_ptr()), P(ixh.data_ptr()), B, kc, slot,
                                    P(u_h.data_ptr()), P(fl_h.data_ptr()))

    def verify_dev():
        psf.ctx.call("qf_synchronize")
        torch.cuda.synchronize()
        assert bool(torch.equal(u, u_ref)) and bool(torch.equal(fl, fl_ref)), "device output differs from the int32 call"
        u.zero_()
        fl.zero_()

    def verify_host():
        uh, fh = u_h[sample], fl_h[sample]
        assert bool(torch.equal(uh, u_ref[sample.to(dev)].cpu())) and bool(torch.equal(fh, fl_ref[sample.to(dev)].cpu())), \
            "host output differs from the int32 call"
        u_h.zero_()
        fl_h.zero_()

    rates = {}
    for rd in range(rounds):
        for t in KEY_COUNTS:
            tb = tables[t]
            psf.ctx.call("qf_ring_set_key_table", P(tb["keys"]), t)
            psf.ctx.call("qf_ring_f_a_keyed_dev", P(sig.data_ptr()), P(tb["idx"].data_ptr()), B, P(u_ref.data_ptr()),
                         P(fl_ref.data_ptr()))
            psf.ctx.call("qf_synchronize")
            assert bool(fl_ref.all())
            for name, mk in (("dev_int32", dev_int32), ("dev_compose", dev_compose), ("dev_fused", dev_fused)):
                dt = timed_dev(torch, mk(tb["idx"]), min_s)
                verify_dev()
                rates.setdefault(f"{name}_T{t}", []).append(B / dt)
                log(f"round {rd} T = {t} {name}: {B / dt / 1e6:.2f} M signatures/s")
            for name, mk in (("host_int32", host_int32), ("host_packed", host_packed)):
                dt = timed_host(mk(tb["idx_h"]), min_s)
                verify_host()
                rates.setdefault(f"{name}_T{t}", []).append(B / dt)
                log(f"round {rd} T = {t} {name}: {B / dt / 1e6:.2f} M signatures/s")
    res["signatures_per_s"] = {k: {"rounds": v, "mean": float(np.mean(v))} for k, v in rates.items()}
    res["chunk"] = "library default (qf_set_chunk not called)"
    res["note"] = ("signatures/s = batch / time of one call over the batch: CUDA events for the dev_* rows, host clock around "
                   "the synchronous host calls for host_* (pinned buffers).  dev_compose includes the decode launch and the "
                   "AND of the canonical flags with the domain flags.  Host-to-device bytes per signature: the row (or slot) "
                   "and its 4-byte key index.")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1), flush=True)


if __name__ == "__main__":
    main()
