"""samp_p throughput for a tagged G-trapdoor key against the identity-tag key (DESIGN.md 4.3).

At C2 (PSFGPV n = 256, q = 2^24, m = 12352) one (A_bar, R) pair gives three keys:
  identity   A = [A_bar | G - A_bar R]                 two-phase recursion
  tagged     A = [A_bar | H G - A_bar R], H random upper unitriangular    two-phase recursion on H^-1 A, targets H^-1 u
  one_pass   the tagged key with QF_DISABLE_TWO_PHASE=1 at trapdoor install (the recursion tagged keys took before)
Device-resident qf_samp_p_dev, 227 328 targets per step, 3 warm-up and 4 timed steps per variant (CUDA events), the
variants alternating twice in the same run; A e = u is checked on every timed output through qf_f_a_dev.  Also times
qf_gen_short_basis against qf_gen_short_basis_tagged and qf_set_trapdoor_gpv for both keys (host clock around calls
that end in a device synchronise).  Prints one JSON line, with the card name and power limit.

--psf perturbation: one C4 shard (PSFPerturbation n = 512, q = 2^32 - 5, m = 32849, r = 9, structured sqrt(Sigma_2)) with
the identity key A = [A_bar | G - A_bar R] and the tagged key [A_bar | H G - A_bar R] of the same (A_bar, R), H random upper
unitriangular (samp_p samples the gadget preimage of H^-1 (u - A p)).  Device-resident qf_samp_p_dev, 60 416 targets per
step (bench.py c4), the two keys alternating as above, A e = u checked through qf_f_a_dev.  Also times the trapdoor install
(qf_set_trapdoor_perturbation, which recognises the tag) for both keys, and qf_set_tag against the full re-install
qf_set_a + qf_set_trapdoor_perturbation that a tag change costs without it.

  python scripts/bench_tagged.py [--psf gpv|perturbation] [--out FILE]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--psf", default="gpv", choices=["gpv", "perturbation"])
    ap.add_argument("--n", type=int, default=None, help="default 256 (gpv), 512 (perturbation)")
    ap.add_argument("--q", type=int, default=None, help="default 2^24 (gpv), 2^32 - 5 (perturbation)")
    ap.add_argument("--batch", type=int, default=None, help="default 227328 (gpv), 60416 (perturbation)")
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    pert = args.psf == "perturbation"
    args.n = args.n or (512 if pert else 256)
    args.q = args.q or (2**32 - 5 if pert else 2**24)
    args.batch = args.batch or (60416 if pert else 227328)
    if pert:
        return main_perturbation(args)

    import tools_b200 as T
    from tools_b200 import _ffi

    info = gpu_info()
    n, q = args.n, args.q
    gp = T.GadgetParameters.init_default(n, q)
    s = float(math.ceil((math.sqrt(gp.m_bar) + 1.0) * math.sqrt(5.0) * math.log2(n)))  # bench.py gpv_s
    rng = np.random.default_rng(1)
    tag = np.triu(rng.integers(0, q, (n, n), dtype=np.int64), 1) + np.eye(n, dtype=np.int64)

    def sync_time(f):
        t0 = time.time()
        f()
        return time.time() - t0

    # ---- keys: the identity key from the device sampler, the tagged key from the same A_bar and R
    ident = T.PSFGPV(gp, s)
    ident.trap_gen(seed=1)  # untimed: module loads
    a_id, r = T.psf._trap_gen_classical(ident, seed=2)
    a_tag = T.psf.gen_trapdoor(gp, a_id[:, : gp.m_bar], r, tag)
    s_id = np.empty((gp.m, gp.m), dtype=np.int64)
    s_tag = np.empty_like(s_id)
    tagged = T.PSFGPV(gp, s)
    tagged._install_a(a_tag)
    tg = np.ascontiguousarray(tag)
    setup = {}
    # warm both entry points once, then time
    ident.ctx.call("qf_gen_short_basis", _ffi.ptr(r), _ffi.ptr(s_id))
    tagged.ctx.call("qf_gen_short_basis_tagged", _ffi.ptr(r), _ffi.ptr(tg), _ffi.ptr(s_tag))
    setup["gen_short_basis_s"] = sync_time(lambda: ident.ctx.call("qf_gen_short_basis", _ffi.ptr(r), _ffi.ptr(s_id)))
    setup["gen_short_basis_tagged_s"] = sync_time(
        lambda: tagged.ctx.call("qf_gen_short_basis_tagged", _ffi.ptr(r), _ffi.ptr(tg), _ffi.ptr(s_tag)))
    td_id, td_tag = (s_id, None), (s_tag, None)
    setup["set_trapdoor_gpv_identity_s"] = sync_time(lambda: ident._install_td(a_id, td_id))
    setup["set_trapdoor_gpv_tagged_s"] = sync_time(lambda: tagged._install_td(a_tag, td_tag))
    os.environ["QF_DISABLE_TWO_PHASE"] = "1"
    one = T.PSFGPV(gp, s)
    one._install_a(a_tag)
    setup["set_trapdoor_gpv_tagged_one_pass_s"] = sync_time(lambda: one._install_td(a_tag, td_tag))
    del os.environ["QF_DISABLE_TWO_PHASE"]
    del s_id, s_tag

    B = args.batch
    rates, checked = throughput(args, {"identity": ident, "tagged": tagged, "one_pass": one}, q, n, gp.m)

    best = {k: max(v) for k, v in rates.items()}
    res = {
        "metric": "samp_p_dev targets/s, tagged vs identity G-trapdoor key",
        "workload": f"PSFGPV n={n} q={q} m={gp.m} s={s}",
        "gpu": info,
        "batch_per_step": B, "warmup_steps": args.warmup, "timed_steps": args.steps, "rounds": args.rounds,
        "rates_per_round": rates,
        "best": best,
        "tagged_over_identity": best["tagged"] / best["identity"],
        "one_pass_over_identity": best["one_pass"] / best["identity"],
        "verified_targets": checked,
        "key_setup_s": setup,
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


def throughput(args, variants, q, n, m):
    """Device-resident qf_samp_p_dev targets/s per variant, variants alternating per round; A e = u and check_domain on
    every timed output through qf_f_a_dev (outside the timed window).  Returns (rates per round, verified targets)."""
    import torch

    from tools_b200 import _ffi

    dev = torch.device("cuda", 0)
    tstream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(tstream)
    lib = _ffi.lib()
    for p in variants.values():
        p.ctx.call("qf_set_stream", _ffi.ptr(tstream.cuda_stream))
    B = args.batch
    u = torch.empty((B, n), dtype=torch.int64, device=dev)
    e = torch.empty((B, m), dtype=torch.int32, device=dev)
    uo = torch.empty_like(u)
    fl = torch.empty(B, dtype=torch.uint8, device=dev)

    def fill(i):
        assert lib.qf_fill_uniform_modq_dev(_ffi.ptr(u.data_ptr()), u.numel(), q, 1000 + i, _ffi.ptr(tstream.cuda_stream)) == 0

    rates = {k: [] for k in variants}
    checked = {k: 0 for k in variants}
    for rnd in range(args.rounds):
        for name, p in variants.items():
            ctx = p.ctx
            for w in range(args.warmup):
                fill(w)
                ctx.call("qf_samp_p_dev", _ffi.ptr(u.data_ptr()), B, 2, w * B, _ffi.ptr(e.data_ptr()))
            ctx.call("qf_synchronize")
            ms = 0.0
            for k in range(args.steps):
                fill(args.warmup + k)
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ev0.record()
                ctx.call("qf_samp_p_dev", _ffi.ptr(u.data_ptr()), B, 2, (args.warmup + k) * B, _ffi.ptr(e.data_ptr()))
                ev1.record()
                ctx.call("qf_synchronize")
                ms += ev0.elapsed_time(ev1)
                ctx.call("qf_f_a_dev", _ffi.ptr(e.data_ptr()), B, _ffi.ptr(uo.data_ptr()), _ffi.ptr(fl.data_ptr()))
                ctx.call("qf_synchronize")
                assert torch.equal(uo, u) and bool(fl.all()), f"{name}: A e != u or check_domain failed"
                checked[name] += B
            rates[name].append(args.steps * B / (ms * 1e-3))
            print(f"round {rnd} {name}: {rates[name][-1] / 1e3:.1f} k/s", file=sys.stderr)
    for p in variants.values():
        p.ctx.call("qf_set_stream", None)
    torch.cuda.set_stream(torch.cuda.default_stream(dev))
    return rates, checked


def main_perturbation(args):
    import tools_b200 as T
    from tools_b200 import gadget

    info = gpu_info()
    n, q, r = args.n, args.q, 9.0
    gp = T.GadgetParameters.init_default(n, q)
    s1 = (math.sqrt(gp.m_bar) + math.sqrt(n * gp.k)) / math.sqrt(2)
    s = float(math.ceil(1.15 * math.sqrt(5 * (s1 * s1 + 1) + 1)))  # bench.py pert_s_for
    rng = np.random.default_rng(1)
    tag = np.triu(rng.integers(0, q, (n, n), dtype=np.int64), 1) + np.eye(n, dtype=np.int64)
    tag2 = np.triu(rng.integers(0, q, (n, n), dtype=np.int64), 1) + np.eye(n, dtype=np.int64)

    def sync_time(f):
        t0 = time.time()
        f()
        return time.time() - t0

    # ---- keys: the identity key from the device sampler, the tagged key from the same A_bar and R; structured
    # sqrt(Sigma_2) (None) and one k x k block of the gadget basis, as PSFPerturbation.trap_gen gives at this size
    ident = T.PSFPerturbation(gp, r, s)
    ident.trap_gen(seed=1)  # untimed: module loads
    a_id, rm = T.psf._trap_gen_classical(ident, seed=2)
    a_bar = np.ascontiguousarray(a_id[:, : gp.m_bar])
    a_tag = T.psf.gen_trapdoor(gp, a_bar, rm, tag)
    blk = gadget.short_basis_gadget_block(gp.k, gp.base, q)
    td = (rm, None, (blk, gadget.gso_small(blk)))
    tagged = T.PSFPerturbation(gp, r, s)
    setup = {"set_trapdoor_identity_s": [], "set_trapdoor_tagged_s": []}
    for _ in range(2):  # the second install of each is the steady-state figure
        for name, p, a in (("identity", ident, a_id), ("tagged", tagged, a_tag)):
            p._install_a(a)
            p._td_id = None
            setup[f"set_trapdoor_{name}_s"].append(sync_time(lambda: p._install_td(a, td)))

    rates, checked = throughput(args, {"identity": ident, "tagged": tagged}, q, n, gp.m)

    # ---- tag switch on the installed tagged key against the full re-install of the switched key
    a_sw = tagged.set_tag(a_tag, td, tag2)  # untimed: first call
    assert np.array_equal(a_sw, T.psf.gen_trapdoor(gp, a_bar, rm, tag2)), "set_tag != gen_trapdoor(A_bar, R, H')"
    sw, cur = [], a_sw
    for i in range(4):
        h = tag if i % 2 == 0 else tag2
        t0 = time.time()
        cur = tagged.set_tag(cur, td, h)
        sw.append(time.time() - t0)
    reinstall = []
    for i in range(2):
        a_new = np.array(a_tag if i % 2 == 0 else a_sw)  # a new array object: _install_a re-installs key and trapdoor
        reinstall.append(sync_time(lambda: (tagged._install_a(a_new), tagged._install_td(a_new, td))))
    setup["set_tag_s"] = sw
    setup["set_a_plus_set_trapdoor_s"] = reinstall

    best = {k: max(v) for k, v in rates.items()}
    res = {
        "metric": "samp_p_dev targets/s, tagged vs identity G-trapdoor key (PSFPerturbation)",
        "workload": f"PSFPerturbation n={n} q={q} m={gp.m} r={r} s={s} structured sqrt(Sigma_2)",
        "gpu": info,
        "batch_per_step": args.batch, "warmup_steps": args.warmup, "timed_steps": args.steps, "rounds": args.rounds,
        "rates_per_round": rates,
        "best": best,
        "tagged_over_identity": best["tagged"] / best["identity"],
        "verified_targets": checked,
        "key_setup_s": setup,
        "set_tag_speedup": min(reinstall) / min(sw),
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
