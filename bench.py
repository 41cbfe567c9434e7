#!/usr/bin/env python3
"""bench.py -- headline benchmark of the scaffolding-MCMC hot path (BASELINE.json metric:
"Delta-log-L proposals scored/sec and MCMC cycle wall-time at pyramid level 4").

A *step* is one MCMC step (= one reference ``step_sampler`` call): <=5 candidate neighbours x <=24
moves scored, the best one applied.  Default workload = BASELINE.json configs[1] (yeast-scale
in-silico assembly, level 4, single chain); ``--workload G`` is configs[3] (~1 Gb synthetic).

  python bench.py --gpus N --steps K --warmup W            our arm (CUDA through the C ABI)
  python bench.py --impl reference ...                     CPU arm: the oracle port of the reference
                                                           algorithm on all host cores
  python bench.py ... --dump-outputs DIR                   also write the timed path's last outputs to DIR/*.npy

Our arm runs the library that build() compiled (``__graft_entry__.build()``) and writes nothing into the tree.

value   = proposals scored / device time (sum of per-step CUDA-event intervals on the launching
          stream; chain state and contacts resident in HBM; L2 flushed between steps, untimed)
e2e     = same metric through the reference-facing facade (``sampler.step_sampler``): host RNG draw
          of the neighbours, ctypes call, H2D of the candidate list and D2H of the result inside the
          timed region (wall clock).
N > 1   = N independent replica chains (different seeds), one process per GPU, NCCL all-gather of
          {likelihood, n_contigs, live scaffold} every ``--gather-every`` steps; weak scaling.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # nothing is written into the tree, which may be read-only
DEFAULT_MODE = "exact"

def params_for(level):
    from instagraal_b200.synth import workload_params
    return workload_params(level)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.rows = []
        self.stop = False
        self.index = index
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self.stop:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([x.strip() for x in out.strip().split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(timeout=6)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 7:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


class stdout_to_stderr:
    """NCCL / torch.distributed print banners to file descriptor 1; the contract is ONE JSON line on stdout"""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)

    def __exit__(self, *a):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_traffic(workload, kernel, mode):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed `ncu --set full` capture of
    this workload (profiles/r2_traffic.json, written by scripts/ncu_traffic.py from the .ncu-rep), or None."""
    p = os.path.join(ROOT, "profiles", "r2_traffic.json")
    try:
        return json.load(open(p)).get("%s/%s/%s" % (workload, mode, kernel))
    except Exception:
        return None


def measure_l2_peak(torch, dev):
    """L2-resident streaming bandwidth of this box: device copy of a 24 MiB buffer (48 MiB footprint << 126 MB L2),
    read + write bytes, best of 20, CUDA events.  The roofline denominator of the workloads whose contacts fit the L2."""
    n = 24 << 20
    a = torch.empty(n, dtype=torch.uint8, device=dev).fill_(1)
    b = torch.empty_like(a)
    for _ in range(5):
        b.copy_(a)
    best = 1e9
    for _ in range(20):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            b.copy_(a)
        e1.record()
        e1.synchronize()
        best = min(best, e0.elapsed_time(e1) / 10.0)
    return 2.0 * n / (best * 1e-3) / 1e9


def build_level(name):
    from instagraal_b200.synth import make_workload
    t0 = time.time()
    level = make_workload(name)
    return level, time.time() - t0


def frag_orders(level, n_chains, n_steps, seed):
    rng = np.random.RandomState(seed)
    out = np.empty((n_chains, n_steps), dtype=np.int32)
    for c in range(n_chains):
        v = []
        while len(v) < n_steps:
            v.extend(rng.permutation(level.n_frags).tolist())
        out[c] = v[:n_steps]
    return out


def dump_outputs(folder, records, rs, best, lik, nc):
    """Writes what the replica pass (the timed path of the headline value) handed its caller after its last step, as
    float64 .npy files, so that two builds run with the same arguments can be compared output for output:
      last_step_<field>[chain]           the last step's record of every chain (ReplicaSet.run_cycle)
      allgather_{best,likelihood,n_contigs}  the exchange that follows it (ReplicaSet.allgather)
      scaffold_<field>[chain, i]         each chain's live scaffold (13 x NF int32) at fragments scaffold_fragment_index[i]:
                                         all of them, or a fixed seeded sample when all chains' full arrays would exceed 48 MB
    With several GPUs the chains are those of rank 0."""
    from instagraal_b200._lib import FIELDS13
    os.makedirs(folder, exist_ok=True)

    def save(name, a):
        np.save(os.path.join(folder, name + ".npy"), np.asarray(a, dtype=np.float64))

    for field in records.dtype.names:
        save("last_step_" + field, records[field][:, -1])
    save("allgather_best", [best])
    save("allgather_likelihood", lik)
    save("allgather_n_contigs", nc)
    nf = rs.nf
    cap = (48 << 20) // (8 * 13 * rs.n)
    idx = np.arange(nf) if nf <= cap else np.sort(np.random.RandomState(0).choice(nf, cap, replace=False))
    states = np.stack([c._get_state()[:, idx] for c in rs.chains])
    save("scaffold_fragment_index", idx)
    for i, field in enumerate(FIELDS13):
        save("scaffold_" + field, states[:, i])


def nuis_stats(s, reset=True):
    import ctypes as C
    from instagraal_b200 import _lib as L
    o = np.zeros(2)
    L.lib().ig_get_nuisance_stats(s._h, o.ctypes.data_as(C.c_void_p), int(reset))
    return float(o[0]), int(o[1])


def single_chain_passes(s, level, args, torch, flush, rank):
    """C4: one chain on one GPU.  Returns the dict of measurements (device-timed steps, per-kernel profile, e2e through
    step_sampler, the same with the nuisance step interleaved as full_em does from cycle 5 on)."""
    dt = np.float32(0.01)
    frs = np.arange(level.n_frags)
    rng = np.random.RandomState(7 + rank)

    def frag_stream(n):
        out = []
        while len(out) < n:
            rng.shuffle(frs)
            out.extend(int(f) for f in frs)
        return out[:n]

    accepted = [0]

    def step_loop(n, nuisance=False, flushing=True):
        for i, f in enumerate(frag_stream(n)):
            if flush is not None and flushing:
                flush.fill_(i & 0xFF)
                torch.cuda.current_stream().synchronize()   # the flush runs on torch's stream, the step on the library's
            s.step_sampler(f, 5, dt)
            if nuisance:
                accepted[0] += int(s.step_nuisance_parameters(dt, i, n)[6])

    res = {}
    # ---- pass 1: device-timed (value of the single-chain configuration)
    step_loop(args.warmup)
    s.set_options(refresh_every=args.refresh_every, use_graph=bool(args.graph))
    s.get_stats(reset=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    step_loop(args.steps)
    torch.cuda.synchronize()
    res["wall_s"] = time.perf_counter() - t0
    st = s.get_stats(reset=True)
    res["dev_ms"], res["proposals"], res["launches"], res["full_refreshes"] = st["ms_step"], st["proposals"], st["launches"], st["full_refreshes"]
    # ---- pass 1b: per-kernel CUDA-event timing for the roofline (profiling on => direct launches, no graph)
    s.set_profiling(True)
    n_prof = min(args.steps, 500)
    step_loop(n_prof)
    res["prof"] = s.get_stats(reset=True)
    res["ktimes"] = s.get_kernel_times(reset=True)
    res["n_prof"] = n_prof
    s.set_profiling(False)
    # ---- pass 2: end to end through the facade (host RNG + ctypes + H2D/D2H), wall clock, no flush (production)
    torch.cuda.synchronize()
    np.random.seed(99 + rank)
    t0 = time.perf_counter()
    step_loop(args.steps, flushing=False)
    torch.cuda.synchronize()
    res["t_e2e"] = time.perf_counter() - t0
    res["prop_e2e"] = s.get_stats(reset=True)["proposals"]
    # ---- pass 3: the same with step_nuisance_parameters after every step (IG:242-252, cycles > 4 of a real run)
    s.param_simu_test = s.param_simu
    p_keep = np.array(list(s.param_simu[0]), dtype=np.float32)
    nuis_stats(s)
    n_nuis = min(args.steps, args.nuisance_steps)
    np.random.seed(299 + rank)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    step_loop(n_nuis, nuisance=True, flushing=False)
    torch.cuda.synchronize()
    res["t_nuis"] = time.perf_counter() - t0
    stn = s.get_stats(reset=True)
    res["prop_nuis"], res["dev_ms_nuis_steps"] = stn["proposals"], stn["ms_step"]
    res["nuis_dev_ms"], res["nuis_calls"] = nuis_stats(s)
    res["n_nuis"] = n_nuis
    res["nuis_accepted"] = accepted[0]
    res["nuis_overlapped"] = int(getattr(s, "n_nuis_overlapped", 0))
    s.set_param_simu(p_keep)   # the random walk of the nuisance parameters must not leak into the next passes
    s.param_simu_test = s.param_simu
    return res


def run_ours(args):
    import torch  # plumbing only: L2 flush buffer, barriers / reductions of the timing numbers, broadcast of the NCCL id
    from instagraal_b200.cuda_lib_gl_single import sampler
    from instagraal_b200.replicas import ReplicaSet, nccl_unique_id

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        with stdout_to_stderr():
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)

    level, t_gen = build_level(args.workload)
    p8 = params_for(level)
    mode = args.mode
    s = sampler(*level.sampler_args(), device=local, rigid_pruning={"exact": 0, "rigid": 1}[mode])
    s.set_param_simu(p8)
    big = level.sparse_matrix.nnz * 8 > 126e6
    burn = args.burn_cycles if args.burn_cycles >= 0 else 2
    t0 = time.time()

    def burnt_state():
        """bomb + `burn` cycles of MCMC (device RNG cycle API): the mid-assembly regime a run spends its time in"""
        np.random.seed(1000)
        s.bomb_the_genome()
        frs = np.arange(level.n_frags)
        for c in range(burn):
            np.random.shuffle(frs)
            s.run_cycle_device(frs, 5, seed=1000, cycle=c)
        return s._get_state()

    st_mid = burnt_state() if args.start in ("bomb", "both") else None
    t_burn = time.time() - t0
    st_true = level.true_state() if args.start in ("true", "both") else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if (args.flush_l2 and not big) else None

    # ---------------- single chain (C2/C3/C4), on rank 0's GPU only when N > 1 is not needed: every rank measures its own
    single = {}
    if world == 1:
        for name, st0 in (("mid", st_mid), ("assembled", st_true)):
            if st0 is None:
                continue
            s._set_state(st0)
            np.random.seed(1000 + rank)
            single[name] = single_chain_passes(s, level, args, torch, flush, rank)
            single[name]["n_contigs_at_start"] = int((st0[0] == 0).sum())
    st_start = st_mid if st_mid is not None else st_true
    start_name = "mid" if st_mid is not None else "assembled"

    # ---------------- replica chains (C5): `--chains` in total, chains / N per GPU, all-gather every gather_every steps
    n_total = args.chains
    n_local = max(1, n_total // world)
    rs = ReplicaSet(s, n_local, seeds=np.arange(rank * n_local, (rank + 1) * n_local, dtype=np.uint64) + 1)
    for c in rs.chains:
        c._set_state(st_start)
        c.set_options(refresh_every=args.refresh_every, use_graph=True)
    nid = None
    if world > 1:
        idt = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            idt = torch.tensor(list(nccl_unique_id()), dtype=torch.uint8, device=dev)
        with stdout_to_stderr():
            dist.broadcast(idt, 0)
        nid = bytes(idt.cpu().tolist())
    with stdout_to_stderr():
        rs.init_comm(rank, world, nid)
        rs.allgather()
    seg = max(1, args.gather_every if args.gather_every > 0 else args.steps // 4)
    warm = frag_orders(level, n_local, min(args.warmup, 200), 5 + rank)
    rs.run_cycle(warm, 5, cycle=100)
    rs.allgather()
    for c in rs.chains:
        c.get_stats(reset=True)
    rs.gather_ms, rs.n_gathers = 0.0, 0
    orders = frag_orders(level, n_local, args.steps, 50 + rank)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    dev_ms_multi, prop_multi, launches = 0.0, 0.0, 0
    with ClockSampler(local) as clk:
        t_wall0 = time.perf_counter()
        for a in range(0, args.steps, seg):
            records = rs.run_cycle(orders[:, a:a + seg], 5, cycle=200 + a)
            sts = [c.get_stats(reset=True) for c in rs.chains]
            dev_ms_multi += max(x["ms_step"] for x in sts)      # the chains of one GPU start together: the slowest one
            prop_multi += float(records["n_proposals"].sum())
            launches += int(sum(x["launches"] for x in sts))
            best, lik, nc = rs.allgather()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        t_wall_multi = time.perf_counter() - t_wall0
    dev_ms_multi += rs.gather_ms
    launches += 3 * n_local * rs.n_gathers

    vals = np.array([dev_ms_multi, prop_multi, t_wall_multi, rs.gather_ms, launches], dtype=np.float64)
    if dist is not None:
        tv = torch.tensor(vals, device=dev)
        mx, sm = tv.clone(), tv.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        dev_ms_max, t_wall_max, gather_ms_max = float(mx[0]), float(mx[2]), float(mx[3])
        prop_sum, launches_sum = float(sm[1]), float(sm[4])
    else:
        dev_ms_max, t_wall_max, gather_ms_max = dev_ms_multi, t_wall_multi, rs.gather_ms
        prop_sum, launches_sum = prop_multi, launches
    if rank != 0:
        rs.free()
        if dist is not None:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, records, rs, best, lik, nc)

    peak, peak_src = measured_peak()
    nnz, ns = s.n_non_zero, int(s.init_n_sub_frags)
    value = prop_sum / (dev_ms_max / 1e3)
    e2e_multi = prop_sum / t_wall_max
    out = {
        "metric": "delta-log-L proposals scored per second (MCMC step_sampler, pyramid level 4)",
        "value": value, "unit": "proposals/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32 expected contacts / f64 log-likelihood accumulation / int32 scaffold",
        "data": "synthetic", "impl": "ours",
        "config": {"workload": args.workload, "n_frags": level.n_frags, "n_sub_frags": ns, "nnz": nnz,
                   "chains": n_local * world, "chains_per_gpu": n_local, "n_neighbours": 5, "mode": mode,
                   "start": start_name, "burn_in_cycles": burn, "n_contigs_at_start": int((st_start[0] == 0).sum()),
                   "l2": ("inputs larger than L2 (%.0f MB of contacts), no flush" % (nnz * 8 / 1e6)) if big else
                         "single-chain passes: flushed between steps with a 256 MiB write (untimed); replica pass: not flushed",
                   "full_likelihood": "maintained incrementally, full recompute every %d steps" % args.refresh_every,
                   "gather_every": seg, "timed": "whole job = %d chains x %d steps + %d all-gathers; time = max over GPUs of "
                                                 "(slowest chain's CUDA-event interval per segment + all-gather events)" % (n_local * world, args.steps, rs.n_gathers)},
        "allgather": {"count": rs.n_gathers, "ms_each_device": gather_ms_max / max(rs.n_gathers, 1), "ms_total": gather_ms_max,
                      "bytes_per_rank": n_local * (64 + 64 * level.n_frags),
                      "what": "ncclAllGather inside the library (ig_allgather_best): {likelihood, n_contigs, 64 B x NF live scaffold} per chain"
                              if world > 1 else "single rank: device copy (no NCCL)"},
        "mcmc_cycle_s": dev_ms_max / 1e3 / args.steps * level.n_frags,
        "proposals_per_step": prop_sum / (n_local * world) / args.steps,
        "wall_s_timed_region": t_wall_max,
        "e2e": {"value": e2e_multi, "unit": "proposals/s",
                "h2d_bytes_per_step": 4, "d2h_bytes_per_step": 56,
                "ms_per_step": t_wall_max / args.steps * 1e3,
                "note": "ReplicaSet.run_cycle -> ig_run_cycles_device_multi with HOST buffers: visiting orders in (4 B per step and chain), "
                        "per-step records out (56 B per step and chain), all-gathers included, wall clock"},
        "gpu_launches": int(launches_sum),
        "clocks": clk.summary(),
        "setup_s": {"generate": t_gen, "burn_in": t_burn},
    }
    # ---------------- single-chain results (C4) + roofline per kernel
    if single:
        scs = {}
        for name, r in single.items():
            stp, n_prof = r["prof"], r["n_prof"]
            n_full = max(stp["full_refreshes"], 0)
            bytes_score = 8 * stp["contacts_read"] + 4 * (stp["rows"] + stp["steps"]) + 16 * stp["rows"] + 32 * stp["frags"]
            bytes_full = 8 * nnz + 4 * (ns + 1) + 20 * ns
            kt = r["ktimes"]
            ms_score = stp["ms_score"] / max(n_prof, 1)
            nuis_ms = r["nuis_dev_ms"] / max(r["nuis_calls"], 1)
            scs[name] = {
                "n_contigs_at_start": r["n_contigs_at_start"],
                "value": r["proposals"] / (r["dev_ms"] / 1e3), "ms_per_step": r["dev_ms"] / args.steps,
                "mcmc_cycle_s": r["dev_ms"] / 1e3 / args.steps * level.n_frags,
                "e2e": {"value": r["prop_e2e"] / r["t_e2e"], "ms_per_step": r["t_e2e"] / args.steps * 1e3,
                        "h2d_bytes_per_step": 40, "d2h_bytes_per_step": 6400,
                        "note": "sampler.step_sampler: host RNG draw, ctypes, 40 B up, one result record down, blocking"},
                "with_nuisance": {"e2e_value": r["prop_nuis"] / r["t_nuis"], "ms_per_step_e2e": r["t_nuis"] / r["n_nuis"] * 1e3,
                                  "mcmc_cycle_s_e2e": r["t_nuis"] / r["n_nuis"] * level.n_frags,
                                  "k_full_lnz_ms_per_call": nuis_ms, "steps": r["n_nuis"],
                                  "proposals_accepted": r["nuis_accepted"], "proposals_prepared_during_the_step": r["nuis_overlapped"],
                                  "note": "step_sampler + step_nuisance_parameters per step (IG:242-252): host fsolve + full likelihood under the test parameters"},
                "without_nuisance_mcmc_cycle_s_e2e": r["t_e2e"] / args.steps * level.n_frags,
                "kernels": {
                    "scoring": {"launches_per_step": "k_stream + k_eval_flat<list> (+ k_score for circular contigs)" if (mode != "exact" and big)
                                                     else ("k_pick + k_eval_flat" if not big else
                                                           "k_stream + k_eval_flat<list> (candidates whose picks fit the list) + k_score (the others)"),
                                "ms_per_step": ms_score, "alg_bytes_per_step": bytes_score / max(n_prof, 1),
                                "achieved_GBs": bytes_score / max(stp["ms_score"], 1e-9) / 1e6,
                                "frac_hbm": bytes_score / max(stp["ms_score"], 1e-9) / 1e6 / peak,
                                "traffic": measured_traffic(args.workload, "scoring", mode + "/" + name)},
                    "k_full_lnz": {"launches": "k_lnz_refresh (rows of the contigs the last move touched) + k_lnz_stream (8 B records of every contact)",
                                   "ms_per_launch": nuis_ms, "alg_bytes_per_launch": bytes_full,
                                   "achieved_GBs": bytes_full / max(nuis_ms, 1e-9) / 1e6,
                                   "frac_hbm": bytes_full / max(nuis_ms, 1e-9) / 1e6 / peak,
                                   "traffic": measured_traffic(args.workload, "k_full_lnz", mode + "/" + name)}},
                "kernel_us_per_step": {k: v / max(n_prof, 1) * 1e3 for k, v in kt.items()},
            }
        out["single_chain"] = scs
        hd = scs[start_name]
        # the top-level object is the SCORING kernels: the only ones of the two that run inside the headline's timed region
        # (step_sampler without the nuisance step) and the ones north_star's roofline target names; the full likelihood of the
        # nuisance step (k_lnz_stream), which takes longer per call at mid-assembly, is listed beside them under "kernels"
        dom = "scoring"
        kd = hd["kernels"][dom]
        out["roofline"] = {"bound": "hbm", "kernel": dom, "state": start_name,
                           "achieved": kd["achieved_GBs"], "peak": peak, "unit": "GB/s", "frac": kd["frac_hbm"],
                           "traffic": kd["traffic"], "peak_source": peak_src,
                           "share_of_step": kd["ms_per_step"] / hd["ms_per_step"],
                           "traffic_source": "profiles/r2_traffic.json: dram__bytes_read + write per step from the committed ncu --set full "
                                             "captures of this workload and state (cold caches: ncu flushes the L2 before every kernel)",
                           "kernels": {st_: scs[st_]["kernels"] for st_ in scs}}
        if not big:
            l2 = measure_l2_peak(torch, dev)
            out["roofline"]["peak_l2_GBs"] = l2
            out["roofline"]["frac_l2"] = kd["achieved_GBs"] / l2
            out["roofline"]["note"] = "this level's contacts fit the 126 MB L2: frac_l2 is against the L2-resident copy bandwidth measured in this run"
    rs.free()
    if not args.no_cpu_baseline and world == 1:
        out["cpu_baseline"] = cpu_baseline(level, p8, st_start, args.cpu_budget_s)
    if not args.no_ref_gpu and world == 1:
        try:
            out["ref_gpu_baseline"] = ref_gpu_baseline(level, p8, st_start, args.ref_gpu_budget_s, local)
            sc_e2e = out["single_chain"][start_name]["e2e"]["value"] if single else None
            if sc_e2e:
                out["ref_gpu_baseline"]["speedup_single_chain_e2e_vs_ref_gpu"] = sc_e2e / out["ref_gpu_baseline"]["value"]
        except Exception as ex:  # the baseline must never break the bench line
            out["ref_gpu_baseline"] = {"unavailable": repr(ex)[:200]}
        try:
            with stdout_to_stderr():   # the reference class logs to stdout
                ri = ref_gpu_baseline_unmodified(level, p8, st_start, args.ref_gpu_budget_s, local)
            out["ref_gpu_baseline_unmodified_class"] = ri
            if single and "value" in ri:
                ri["speedup_single_chain_e2e_vs_ref_gpu"] = out["single_chain"][start_name]["e2e"]["value"] / ri["value"]
        except Exception as ex:
            out["ref_gpu_baseline_unmodified_class"] = {"unavailable": repr(ex)[:300]}
    print(json.dumps(out))
    if dist is not None:
        dist.destroy_process_group()


def _oracle_chain(level, p8, state13, seed, budget_s, max_steps=None, warm=0):
    from oracle.sampler_oracle import OracleSampler
    from instagraal_b200._lib import FIELDS13
    o = OracleSampler(level, p8)
    if state13 is not None:
        o.live = {k: state13[i].copy() for i, k in enumerate(FIELDS13)}
    np.random.seed(seed)
    frs = np.arange(level.n_frags)
    np.random.shuffle(frs)
    for f in frs[:warm]:
        o.step_sampler(int(f), 5)
    t0 = time.perf_counter()
    n_prop = n_steps = 0
    for f in frs[warm:]:
        o.step_sampler(int(f), 5)
        n_prop += int(sum(o.n_uniq_list))
        n_steps += 1
        if time.perf_counter() - t0 > budget_s or (max_steps is not None and n_steps >= max_steps):
            break
    return n_prop, n_steps, time.perf_counter() - t0


def cpu_baseline(level, p8, state13, budget_s):
    """the oracle (NumPy port of the reference algorithm) on one host core, bounded sample"""
    n_prop, n_steps, dt = _oracle_chain(level, p8, state13, 3, budget_s)
    return {"value": n_prop / dt, "unit": "proposals/s", "cores": 1, "kind": "port",
            "sample": "%d step_sampler calls (%d proposals) of the same workload from the same burnt-in scaffold, %.1f s"
                      % (n_steps, n_prop, dt)}


def ref_gpu_baseline(level, p8, state13, budget_s, device=0):
    """B-ref (GPU): the reference's own kernels (oracle/_ref/ref_kernels.cubin) driven in the reference's
    launch order with its per-launch synchronisation, NumPy 'thrust' round trips, 17-array D2H copies
    and Python dist loop (oracle/ref_replay.py, validated against the golden vectors on the CPU backend)."""
    cubin = os.path.join(ROOT, "oracle", "_ref", "ref_kernels.cubin")
    if not os.path.exists(cubin):
        return {"unavailable": "oracle/_ref/ref_kernels.cubin not built"}
    from oracle.ref_replay import RefReplaySampler
    from oracle.sampler_oracle import return_neighbours, setup_distri_frags
    r = RefReplaySampler(level, p8, backend="gpu", device=device)
    if state13 is not None:
        r.set_state(state13)
    distri = setup_distri_frags(level.sub_sampled_sparse_matrix, level.n_frags)
    np.random.seed(3)
    frs = np.arange(level.n_frags)
    np.random.shuffle(frs)
    r.step_sampler(int(frs[0]), return_neighbours(distri, level.n_frags, int(frs[0]), 5))  # warm-up (module load, caches)
    l0 = r.be.n_launch
    t0 = time.perf_counter()
    n_prop = n_steps = 0
    for f in frs[1:]:
        r.step_sampler(int(f), return_neighbours(distri, level.n_frags, int(f), 5))
        n_prop += int(sum(r.n_uniq_list))
        n_steps += 1
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return {"value": n_prop / dt, "unit": "proposals/s", "ms_per_step": dt / n_steps * 1e3, "steps": n_steps,
            "kernel_launches_per_step": (r.be.n_launch - l0) / n_steps,
            "kind": "reference kernels (cubin built from /root/reference) + restated reference host sequence (route ii)",
            "sample": "%d step_sampler calls from the same burnt-in scaffold, %.1f s" % (n_steps, dt)}


def ref_gpu_baseline_unmodified(level, p8, state13, budget_s, device=0):
    """B-ref (GPU), route (i): the UNMODIFIED reference sampler class (verbatim copy under baseline/_ref) on this GPU through
    oracle/ref_harness_gpu, a stand-in for pycuda over cuda-python; its own return_neighbours, its own step_sampler."""
    from oracle import ref_unmodified as ru
    if not ru.available():
        return {"unavailable": "baseline/_ref/instagraal or oracle/_ref/ref_kernels.cubin not built"}
    t0 = time.perf_counter()
    r = ru.UnmodifiedSampler(level, p8, device=device)
    t_ctor = time.perf_counter() - t0
    if state13 is not None:
        r.set_state(state13)
    np.random.seed(3)
    frs = np.arange(level.n_frags)
    np.random.shuffle(frs)
    r.step_sampler(int(frs[0]))   # warm-up
    l0 = r.n_launch
    t0 = time.perf_counter()
    n_prop = n_steps = 0
    for f in frs[1:]:
        r.step_sampler(int(f))
        n_prop += int(np.count_nonzero(r.all_scores))
        n_steps += 1
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return {"value": n_prop / dt, "unit": "proposals/s", "ms_per_step": dt / n_steps * 1e3, "steps": n_steps,
            "kernel_launches_per_step": (r.n_launch - l0) / n_steps, "constructor_s": t_ctor,
            "kind": "unmodified reference sampler class (baseline/_ref copy) + pycuda stand-in over cuda-python + reference cubin (route i)",
            "sample": "%d step_sampler calls from the same burnt-in scaffold, %.1f s" % (n_steps, dt)}


_REF_LEVEL = None


def _ref_worker(a):
    seed, budget, max_steps, warm = a
    level = _REF_LEVEL   # built once in the parent, inherited through fork (copy-on-write)
    p8 = params_for(level)
    return _oracle_chain(level, p8, None, seed, budget, max_steps, warm)


def run_reference(args):
    """CPU arm: the reference's algorithm (oracle port: NumPy transcription of its kernels + its orchestration) on every
    host core, one independent chain per process.  A "step" of this arm is one step_sampler call on every core; at most
    --steps of them are timed after min(--warmup, 2) untimed ones, and the sample is cut at --cpu-budget-s seconds so the
    run stays bounded whatever K is (at the 1 Gb level one call takes tens of seconds: every core then times one call)."""
    global _REF_LEVEL
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    budget = max(5.0, min(args.cpu_budget_s, 60.0))
    level, _ = build_level(args.workload)
    _REF_LEVEL = level
    big = level.sparse_matrix.nnz > 20e6
    n_proc = min(cores, 8) if big else cores   # ~6 GB of temporaries per worker at the 1 Gb level
    t0 = time.perf_counter()
    with mp.get_context("fork").Pool(n_proc) as pool:
        warm = 0 if big else max(0, min(args.warmup, 2))
        res = pool.map(_ref_worker, [(100 + i, budget, args.steps, warm) for i in range(n_proc)])
    wall = time.perf_counter() - t0
    n_prop = sum(r[0] for r in res)
    n_steps = sum(r[1] for r in res)
    t_max = max(r[2] for r in res)
    v = n_prop / t_max
    out = {
        "metric": "delta-log-L proposals scored per second (MCMC step_sampler, pyramid level 4)",
        "value": v, "unit": "proposals/s", "n_gpus": int(os.environ.get("WORLD_SIZE", "1")),
        "steps": max(r[1] for r in res), "warmup": warm, "requested_steps": args.steps, "requested_warmup": args.warmup,
        "ms_per_step": t_max / max(n_steps / n_proc, 1) * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32 expected contacts / f64 accumulation / int32 scaffold", "data": "synthetic",
        "impl": "reference",
        "config": {"workload": args.workload, "n_frags": level.n_frags, "n_sub_frags": level.n_sub_frags,
                   "nnz": int(level.sparse_matrix.nnz - np.count_nonzero(level.sparse_matrix.diagonal())),  # strict upper, as the GPU arm counts
                   "chains": n_proc, "n_neighbours": 5,
                   "note": "the reference is GPU-only (pycuda); this arm is its algorithm transcribed to NumPy (oracle/), "
                           "one chain per host process from the contig-order start (the synthetic assembly's initial contigs: the "
                           "regime of the GPU arm's mid-assembly state, which itself lies 2 MCMC cycles of this arm away: weeks on the host at the 1 Gb level)"},
        "cpu_baseline": {"value": v, "unit": "proposals/s", "cores": n_proc, "kind": "port",
                         "sample": "%d processes x <= %.0f s of step_sampler calls (%d steps, %d proposals), wall %.1f s"
                                   % (n_proc, budget, n_steps, n_prop, wall)},
        "e2e": {"value": v, "unit": "proposals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="G", help="G = BASELINE.json configs[3] (~1 Gb, the config the metric is quoted on); T, Y3, yeast_toy")
    ap.add_argument("--chains", type=int, default=8, help="replica chains in total (configs[4]: 8), split evenly over the GPUs")
    ap.add_argument("--burn-cycles", type=int, default=-1)
    ap.add_argument("--start", default="both", choices=["bomb", "true", "both"],
                    help="single-chain passes from the mid-assembly state (bomb + burn-in), the fully assembled one, or both")
    ap.add_argument("--flush-l2", type=int, default=1)
    ap.add_argument("--gather-every", type=int, default=0, help="steps between all-gathers (0: steps / 4)")
    ap.add_argument("--refresh-every", type=int, default=4096)
    ap.add_argument("--graph", type=int, default=1)
    ap.add_argument("--mode", default=DEFAULT_MODE, choices=["exact", "rigid"],
                    help="exact: reproduce the reference's float32 re-rounding of rigidly shifted coordinates bit for bit; "
                         "rigid: skip contacts whose two ends move together (DESIGN.md D2)")
    ap.add_argument("--nuisance-steps", type=int, default=500)
    ap.add_argument("--cpu-budget-s", type=float, default=20.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-gpu", action="store_true")
    ap.add_argument("--ref-gpu-budget-s", type=float, default=10.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed replica pass returned after its last step to DIR/<name>.npy (rank 0's chains)")
    args = ap.parse_args()
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
