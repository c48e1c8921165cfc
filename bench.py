#!/usr/bin/env python
"""bench.py — the judged benchmark of the idle-decision hot path.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # the CPU restatement (reference arm)
    torchrun --nproc-per-node N ... bench.py --gpus N ...     # N > 1: one rank per GPU
    python bench.py ... --dump-outputs DIR                     # + the last timed step's outputs as DIR/*.npy

Workload (BASELINE.json configs[1], the configuration the metric is quoted on that fits one GPU):
10,000 pods x 4 GPUs x 1,800 samples (30 min @ 1 s) of synthetic DCGM_FI_DEV_GPU_UTIL per B200,
f32, with the 5 %-ineligible age/phase gate.  At N > 1 the pod axis is sharded (weak scaling:
one such window per rank) and every step ends with ONE exchange of the packed decision bitmap
(fused into the fold kernel over NVLink peer memory; --collective nccl = one ncclAllGather).
A "step" = one pass of the hot path over one window: window reduction (max over time per
series), `== 0`, ANY-GPU fold, gate, packed bitmap (+ exchange).

Metric: DCGM samples reduced per second, whole job (pod-decisions/s reported beside it).
  value : windows already resident in HBM (4 distinct windows rotated, 1.15 GB >> 126 MB L2);
          EXACTLY K steps in one region, CUDA events on the engine's stream, max over ranks.
          Everything host-side (batch marshalling, clock sampler) happens BEFORE the barrier and the
          region opens with a device-side rendezvous of all ranks (gpr_timer_begin), so rank start
          skew is not part of anybody's timed region.
  per_step : median / p95 of the K per-step device times (%globaltimer stamps written by the fold
          kernel when a decision completes), max over ranks — SURVEY.md §8(d)'s definition, reported
          beside the contiguous figure.
  e2e   : the same step through the blocking C-ABI call gpr_decide() with the window in PINNED
          HOST memory: H2D of the window + gates and D2H of the bitmap + counts inside the timing.
  parity: the gathered bitmap of the step before the timed region AND of the last timed step, and the
          summed counts, against the CPU oracle over all N x 10,000 pods (checker only, after timing).
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SEED = 0x5EED0002
PODS, GPUS, SAMPLES = 10000, 4, 1800
ROTATE = 4
METRIC, UNIT = "dcgm_samples_reduced_per_sec", "samples/s"


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def recorded_traffic():
    """dram bytes per launch of the dominant kernel from the committed ncu --set full capture
    (a STATIC record: it is not re-measured by this run; `traffic_source` in the line says so)"""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        return None


class ClockSampler:
    """polls SM clock + throttle reasons through NVML while the timed regions run"""

    def __init__(self, index):
        self.index, self.samples, self.stop_flag, self.t = index, [], threading.Event(), None
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        while not self.stop_flag.is_set():
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                util = nv.nvmlDeviceGetUtilizationRates(self.h).gpu
                self.samples.append((mhz, reasons, util))
            except Exception:
                pass
            time.sleep(0.02)

    def start(self):
        if self.nv:
            self.t = threading.Thread(target=self._loop, daemon=True)
            self.t.start()

    def stop(self):
        self.stop_flag.set()
        if self.t:
            self.t.join()
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
                 0x4: "sw_power_cap", 0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting",
                 0x100: "display_clock_setting", 0x10: "sync_boost"}
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        mhz = sorted(s[0] for s in self.samples)
        seen = 0
        for s in self.samples:
            seen |= s[1]
        return {"sm_mhz": mhz[len(mhz) // 2], "sm_max_mhz": self.max_mhz,
                "reasons": sorted(n for b, n in names.items() if seen & b), "samples": len(self.samples)}


def workload_config(world):
    """identical in both arms (the driver compares the two `config` objects)"""
    return {"workload": f"C2 (BASELINE configs[1]): {PODS} pods x {GPUS} GPUs x {SAMPLES} samples "
                        f"(30 min @ 1 s) per B200, util plane + age/phase gate",
            "pods_per_gpu": PODS, "gpus_per_pod": GPUS, "samples_per_series": SAMPLES,
            "bytes_per_step_per_gpu": 4 * PODS * GPUS * SAMPLES, "seed": hex(SEED),
            "sharding": f"pod axis, {world} rank(s), one exchange of the packed bitmap per step"
                        if world > 1 else "single GPU",
            "l2": f"{ROTATE} distinct 288 MB windows rotated (1.15 GB vs 126 MB L2), no flush needed"}


# ---------------------------------------------------------------------------------------------
# reference arm: the CPU restatement on the box's host cores
# ---------------------------------------------------------------------------------------------
def cpu_pass_factory(n_threads):
    """returns run(step_index, pods) over ROTATE distinct C2 windows held in host RAM (1.15 GB in total,
    like the GPU arm, so that no arm is timed out of a last-level cache).  The pool's workers are pinned
    to distinct CPUs and fill the windows with the same pod split they later reduce (NUMA-local pages):
    the baseline gets its best shot."""
    import numpy as np
    from oracle import oracle_c
    lib = oracle_c.load()
    oracle_c.pool_pin(True)
    wins = [(oracle_c.synth_fill(SEED + 16 * i, 0, 0, PODS, GPUS, SAMPLES, n_threads),
             oracle_c.synth_eligible(SEED + 16 * i, 0, PODS)) for i in range(ROTATE)]
    W = (PODS + 31) // 32
    dbits = np.zeros(W, np.uint32)
    cbits = np.zeros(W, np.uint32)
    counts = np.zeros(3, np.uint64)

    def run(i=0, pods=PODS, threads=n_threads):
        u, e = wins[i % ROTATE]
        rc = lib.gpo_decide_mt(threads, u.ctypes.data, None, e.ctypes.data, None, 0, pods, GPUS,
                               SAMPLES, 0, 0.0, dbits.ctypes.data, cbits.ctypes.data, None,
                               counts.ctypes.data)
        assert rc == 0
    return run, dbits, counts


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0  # under torchrun only rank 0 measures the CPU arm
    from oracle import oracle_c
    n_threads = oracle_c.hardware_threads()
    run, dbits, counts = cpu_pass_factory(n_threads)
    run(0)
    t0 = time.perf_counter()
    run(1)
    one = time.perf_counter() - t0
    # bound the whole run to ~150 s: shrink the per-step sample if the full window is too slow
    reps = 7
    pods = PODS
    budget = 150.0
    if one * (args.steps * reps + args.warmup) > budget:
        reps = max(3, min(reps, int(budget / (one * args.steps))))
    if one * (args.steps * reps + args.warmup) > budget:
        pods = max(32, int(PODS * budget / (one * (args.steps * reps + args.warmup))) // 32 * 32)
    for i in range(args.warmup):
        run(i, pods)
    # the CPU arm is the baseline: time `reps` repetitions of the K steps and report the BEST one
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        for i in range(args.steps):
            run(i, pods)
        times.append(time.perf_counter() - t0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dbits[:(pods + 31) // 32], counts)
    dt = min(times)
    samples = pods * GPUS * SAMPLES
    value = samples * args.steps / dt
    sample_desc = (f"{pods} of {PODS} pods x {GPUS} x {SAMPLES} per step ({samples * 4 / 1e6:.0f} MB), "
                   f"{ROTATE} windows rotated in host RAM, {n_threads} pinned POSIX threads over contiguous pod "
                   f"ranges (NUMA-local first touch), best of {reps} repetitions of the {args.steps} steps")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT,
        "pod_decisions_per_sec": pods * args.steps / dt,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": n_threads, "kind": "port",
                         "sample": sample_desc,
                         "host_stream_gbs": value * 4 / 1e9,
                         "repetitions_ms_per_step": [round(t / args.steps * 1e3, 4) for t in times]},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "reference = CPU restatement (oracle/gpr_oracle.c) of the PromQL the reference ships "
                "to Prometheus; the Rust reference cannot be built here and does no arithmetic itself. "
                "At N > 1 rank 0 alone runs it: one C2 window per step = a 1/N sample of the N-GPU workload",
    }
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------------------
# CUDA arm
# ---------------------------------------------------------------------------------------------
def step_stats(durations_us):
    import numpy as np
    d = np.sort(np.asarray(durations_us, dtype=np.float64))
    if d.size == 0:
        return {"median_us": None, "p95_us": None, "min_us": None, "max_us": None}
    return {"median_us": float(np.median(d)), "p95_us": float(d[min(d.size - 1, int(np.ceil(0.95 * d.size)) - 1)]),
            "min_us": float(d[0]), "max_us": float(d[-1])}


def dump_outputs(out_dir, decision_bits, counts):
    """what a caller of the timed path receives from its last step, as float64 (exact for uint32 words):
    decision_bits.npy = the packed per-pod idle bitmap (rank-major words at N > 1), counts.npy =
    [n_series, n_candidates, n_decisions] summed over ranks"""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "decision_bits.npy"), np.asarray(decision_bits, np.uint32).astype(np.float64))
    np.save(os.path.join(out_dir, "counts.npy"), np.asarray(counts, np.float64))


def run_cuda(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import gpu_pruner_b200 as g

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch N > 1 with torch.distributed.run (one rank per GPU)")
        args.gpus = world
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback "
                         "(use --impl reference for the CPU restatement)")
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(dev))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def reduce_sum_i(xs):
        t = torch.tensor(list(xs), dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [int(v) for v in t.tolist()]

    sh = g.shard_pods(PODS * world, rank, world) if world > 1 else g.Shard(0, 1, PODS, PODS, 0, PODS)
    P, G, T = sh.pods_per_rank, GPUS, SAMPLES
    profiling_only = bool(args.strong_total)      # c4 / c5: device-resident timing only
    eng = g.IdleEngine(device=local, max_pods=0 if profiling_only else P, max_gpus=G, max_samples=T,
                       kernel=args.kernel)
    if world > 1 and args.collective == "p2p":
        # fused: the fold kernel itself pushes the words to the peers over NVLink.  If peer mapping is
        # not possible on this box (all ranks must agree), use the NCCL allgather instead.
        ok = 1
        try:
            handles = [None] * world
            dist.all_gather_object(handles, eng.p2p_init(rank, world, P))
            eng.p2p_attach(handles)
        except g.GprError as ex:
            ok = 0
            print(f"[rank {rank}] peer-memory exchange unavailable ({ex}); falling back to ncclAllGather",
                  file=sys.stderr)
        flag = torch.tensor([ok], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0:
            if ok:   # this rank attached but another could not: start over without the fused exchange
                eng.close()
                eng = g.IdleEngine(device=local, max_pods=0 if profiling_only else P, max_gpus=G,
                                   max_samples=T, kernel=args.kernel)
            args.collective = "nccl"
    if world > 1 and args.collective == "nccl":
        uid = [eng.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        eng.comm_init(uid[0], rank, world)

    # ---- synthetic windows, generated on the owning GPU (no scatter) --------------------------
    wins = []
    for i in range(ROTATE):
        u = torch.full((P, G, T), float("nan"), dtype=torch.float32, device=dev)
        e = torch.zeros(P, dtype=torch.uint8, device=dev)
        torch.cuda.synchronize()   # torch's fills first: the engine's stream is not ordered with torch's
        eng.synth_fill(SEED + 16 * i, 0, u, sh.pod_begin, sh.pods_real, G, T)
        eng.synth_eligible(SEED + 16 * i, e, sh.pod_begin, sh.pods_real)
        wins.append((u, e))
    W_rank = (P + 31) // 32
    W_out = W_rank * world
    dbits = torch.zeros(W_out, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()

    def step(i, blocking=False):
        u, e = wins[i % ROTATE]
        return eng.decide_ptr(u, P, G, T, dbits, eligible=e, blocking=blocking)

    def global_bits():
        return dbits.cpu().numpy().view(np.uint32).copy()

    # One blocking step on window 0 before the timed region; its (global) bitmap is kept for the
    # parity check after the timing.  Every rank takes the step: with an exchange attached it is collective.
    r = step(0, blocking=True)
    first_bits = global_bits()
    first_counts = reduce_sum_i((int(r.n_series), int(r.n_candidates), int(r.n_decisions)))
    n_words_mine = (sh.pods_real + 31) // 32
    my_bits0 = first_bits[rank * W_rank: rank * W_rank + n_words_mine].copy()

    # ---- timed region 1: windows resident in HBM ------------------------------------------------
    # one pre-marshalled batch of decisions per C-ABI call (gpr_decide_batch_async): the timed loop
    # contains no per-step Python, only the library's own launch path.  Everything Python does is done
    # BEFORE the barrier; gpr_timer_begin then aligns the ranks on the device.
    chunk = 200                                   # the async result ring holds 256 entries
    batch = eng.make_batch([dict(util=wins[i % ROTATE][0], eligible=wins[i % ROTATE][1], P=P, G=G, T=T,
                                 decision_bits=dbits) for i in range(min(chunk, max(args.steps, 1)))])
    sampler = ClockSampler(local)
    for i in range(args.warmup):
        step(i)
    eng.sync()
    sampler.start()

    phases = []

    def timed_pass(n_steps):
        """K steps in chunks; returns (device ms, per-step durations in us, launches, last results array,
        steps in the last chunk)"""
        ms, durs, done, launches, ress, n = 0.0, [], 0, 0, None, 0
        while done < n_steps:
            n = min(chunk, n_steps - done)
            l0 = eng.launch_count()
            eng.timer_begin()                     # device-side rendezvous of all ranks + start event
            ress = eng.decide_batch_async(batch, n)
            ms += eng.timer_end()
            eng.sync()
            launches += eng.launch_count() - l0 - 1   # the rendezvous kernel is outside the event pair
            t0, st = eng.step_stamps()
            durs.extend(np.diff(np.concatenate([np.array([t0], np.uint64), st]).astype(np.int64)) / 1e3)
            ph = eng.phase_stamps().astype(np.int64)
            if len(ph) == len(st):      # fold kernel phases of every step: start -> folded -> flags raised -> peers in -> done
                phases.append(np.stack([ph[:, 1] - ph[:, 0], ph[:, 2] - ph[:, 1], ph[:, 3] - ph[:, 2],
                                        st.astype(np.int64) - np.where(ph[:, 3] > 0, ph[:, 3], ph[:, 1])], axis=1) / 1e3)
            done += n
        return ms, durs, launches, ress, n

    barrier()
    ms_dev, durs, launches, ress, n_last = timed_pass(args.steps)
    barrier()
    ms_total = reduce_max(ms_dev)
    ms_per_step = ms_total / args.steps
    st = step_stats(durs)
    per_step = {k: (reduce_max(v) if v is not None else None) for k, v in st.items()}
    per_step["first_us"] = reduce_max(float(durs[0])) if len(durs) else None
    per_step["first_steps_us_rank0"] = [round(float(x), 2) for x in durs[:8]]
    if phases:
        ph = np.concatenate(phases)[:args.steps]
        med = np.median(ph, axis=0)
        per_step["fold_kernel_phases_us"] = {
            "fold": reduce_max(float(med[0])), "push_and_fence": reduce_max(float(med[1])) if world > 1 else None,
            "wait_for_peers": reduce_max(float(med[2])) if world > 1 else None, "assemble_and_publish": reduce_max(float(med[3])),
            "note": "median over the timed steps of the first pass, max over ranks; the fold kernel's critical path per step"}
    per_step["note"] = ("device %globaltimer stamps written by the fold kernel when a decision (exchange "
                        "included) completes; differences of consecutive stamps; each statistic is the max over ranks")
    # the LAST timed step's global bitmap and counts (catches a stale double buffer under PDL overlap)
    last_window = (n_last - 1) % ROTATE
    last_bits = global_bits()
    last_counts = reduce_sum_i((int(ress[n_last - 1].n_series), int(ress[n_last - 1].n_candidates),
                                int(ress[n_last - 1].n_decisions)))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_bits, last_counts)

    # ---- N > 1: where the step time goes (fused exchange only) ------------------------------------
    breakdown = None
    if world > 1 and args.collective == "p2p" and not args.no_breakdown:
        breakdown = {}
        for name, mode in (("no_exchange", 2), ("push_only", 1), ("full", 0)):
            barrier()
            eng.p2p_debug(mode)
            m, d, _, _, _ = timed_pass(args.steps)
            breakdown[name + "_us_per_step"] = reduce_max(m) / args.steps * 1e3
            breakdown[name + "_median_us"] = reduce_max(step_stats(d)["median_us"])
        eng.p2p_debug(0)
        barrier()
        breakdown["note"] = ("same K steps re-timed with gpr_p2p_debug: 2 = fold without peer stores, 1 = peer stores + "
                             "flags but no wait, 0 = the full exchange (a second sample of `ms_per_step`)")

    # for transparency: device time of ONE isolated blocking decision (no overlap with a neighbour)
    iso = sorted(step(i, blocking=True).kernel_ms for i in range(15))
    single_decision_us = iso[len(iso) // 2] * 1e3
    barrier()
    real_pods_total = PODS * world
    samples_per_step = real_pods_total * G * T
    value = samples_per_step / (ms_per_step * 1e-3)

    e2e_s_per_step, e2e_ok, e2e_steps = float("nan"), True, 0
    e2e_u8 = None
    pcie = None
    h_u = h_e = None
    if not profiling_only:
        # ---- timed region 2: end to end through gpr_decide() with pinned HOST buffers ----------------
        e2e_steps = max(1, min(args.steps, args.e2e_steps))
        h_u = eng.host_array((P, G, T), np.float32)
        h_e = eng.host_array((P,), np.uint8)
        h_bits = eng.host_array((max(W_out, 1),), np.uint32)
        eng.memcpy(h_u, wins[0][0], h_u.nbytes, 0, 1)
        eng.memcpy(h_e, wins[0][1], h_e.nbytes, 0, 1)

        def e2e_step():
            return eng.decide_ptr(h_u, P, G, T, h_bits, eligible=h_e, in_kind=0, out_kind=0, blocking=True)

        for _ in range(3):
            r = e2e_step()
        # the host-window path must reproduce the device-window bitmap of the same window
        e2e_ok = bool(np.array_equal(h_bits[:W_out], first_bits))
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        torch.cuda.synchronize()
        e2e_s_per_step = reduce_max(time.perf_counter() - t0) / e2e_steps
        barrier()
        # the PCIe roofline of that call: a plain pinned H2D copy of the same 288 MB (best of 5)
        scratch = eng.device_alloc(h_u.nbytes)
        best = float("inf")
        for _ in range(5):
            t0 = time.perf_counter()
            eng.memcpy(scratch, h_u, h_u.nbytes, 1, 0)
            best = min(best, time.perf_counter() - t0)
        eng.device_free(scratch)
        h2d_peak = h_u.nbytes / best / 1e9
        pcie = {"h2d_gbs": (h_u.nbytes + h_e.nbytes) / e2e_s_per_step / 1e9, "h2d_peak_gbs": h2d_peak,
                "pcie_frac": (h_u.nbytes + h_e.nbytes) / e2e_s_per_step / 1e9 / h2d_peak,
                "peak_source": "blocking cudaMemcpy of the same pinned 288 MB window on this rank, best of 5"}

        # ---- extra: the same call with the window in the compact wire format (GPR_FMT_U8B, one
        # byte per sample; DCGM_FI_DEV_GPU_UTIL is an integer percentage) — reported beside `e2e`,
        # never instead of it
        if world == 1:
            h_u8 = eng.host_array((P, G, T), np.uint8)
            np.copyto(h_u8, np.where(np.isnan(h_u), 0, h_u + 1), casting="unsafe")
            h_bits8 = eng.host_array((max(W_out, 1),), np.uint32)

            def e2e_u8_step():
                return eng.decide_ptr(h_u8, P, G, T, h_bits8, eligible=h_e, in_kind=0, out_kind=0,
                                      blocking=True, util_format=g.ffi.GPR_FMT_U8B)

            for _ in range(3):
                e2e_u8_step()
            u8_ok = bool(np.array_equal(h_bits8[:n_words_mine], my_bits0))
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                e2e_u8_step()
            torch.cuda.synchronize()
            dt8 = (time.perf_counter() - t0) / e2e_steps
            e2e_u8 = {"value": samples_per_step / dt8, "unit": UNIT, "pod_decisions_per_sec": PODS / dt8,
                      "ms_per_step": dt8 * 1e3, "steps": e2e_steps,
                      "h2d_bytes_per_step": int(h_u8.nbytes + h_e.nbytes), "d2h_bytes_per_step": int(W_out * 4 + 24),
                      "api": "gpr_decide(ctx, window{mem_kind=HOST, util_format=GPR_FMT_U8B}, result{HOST})",
                      "matches_device_path": u8_ok}
            e2e_ok = e2e_ok and u8_ok

    # ---- extra: daemon steady state (--daemon-mode, --check-interval 180 s): the window stays
    # resident in HBM, a tick moves only the 180 new columns per series across PCIe and rescans.
    resident = None
    if world == 1 and not profiling_only:
        n_new = 180
        eng.resident_init(P, G, T)
        u_ptr, _, _ = eng.resident_planes()
        eng.synth_fill(SEED, 0, u_ptr, 0, P, G, T)
        h_cols = eng.host_array((P, G, n_new), np.float32)
        h_cols[:] = 0.0
        rbits = eng.host_array((max(W_out, 1),), np.uint32)

        def tick():
            eng.append(h_cols, None, n_new)
            return eng.decide_ptr(None, 0, 0, 0, rbits, eligible=h_e, in_kind=0, out_kind=0, resident=True)

        for _ in range(3):
            tick()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            tick()
        torch.cuda.synchronize()
        dt_r = (time.perf_counter() - t0) / e2e_steps
        resident = {"value": samples_per_step / dt_r, "unit": UNIT, "pod_decisions_per_sec": PODS / dt_r,
                    "ms_per_tick": dt_r * 1e3, "steps": e2e_steps,
                    "h2d_bytes_per_step": int(h_cols.nbytes + h_e.nbytes), "d2h_bytes_per_step": int(W_out * 4 + 24),
                    "api": "gpr_append(180 new columns / series, pinned host) + gpr_decide_resident()",
                    "note": "steady-state tick of daemon mode: the 30-min window is resident in HBM, only the "
                            "columns scraped since the previous tick (check-interval 180 s @ 1 s) cross PCIe"}
    clocks = sampler.stop()

    # ---- extra: the same steady-state tick through the PRODUCT BINARY (gpu-pruner -d): tick 0 parses the full range
    # query (1.25 GB of response text) on the GPU into the resident ring, later ticks parse only the 180 s scraped
    # since (135 MB of text) into it and rescan.  Fixture files stand in for the Prometheus HTTP responses; the time
    # to read them from disk is reported separately and not counted.
    daemon_binary = None
    if world == 1 and not profiling_only and not args.no_daemon_binary:
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import daemon_ticks_bench
            eng.sync()
            d = daemon_ticks_bench.run(PODS, G, T, 180, ticks=4, cpu_ticks=0)
            tk = d["resident"]["ticks"]
            daemon_binary = {
                "steady_tick_ms": d["resident"].get("steady_tick_ms_median"), "unit": "ms per tick, response text in host memory -> verdict",
                "value": d["resident"].get("samples_per_s_at_median_tick"), "value_unit": UNIT,
                "first_tick_ms": tk[0].get("engine_ms") if tk else None, "text_bytes": d["text_bytes"],
                "ticks": tk, "steady_note": d["resident"]["steady_note"],
                "api": "gpu-pruner -d (C++ host): gpr_text_scan_begin/_next + gpr_resident_advance + "
                       "gpr_text_parse(GPR_TEXT_RESIDENT) + gpr_decide_resident"}
        except Exception as ex:  # an extra must never take the judged line down
            daemon_binary = {"error": repr(ex)[:300]}

    parity_failed = False
    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        bytes_per_launch = 4.0 * P * G * T          # algorithmic: 4 B per sample, read once
        achieved = bytes_per_launch / (ms_per_step * 1e-3) / 1e9
        traffic = recorded_traffic()
        kname = args.kernel if args.kernel != "auto" else "tma"
        line = {
            "metric": METRIC, "value": value, "unit": UNIT,
            "pod_decisions_per_sec": real_pods_total / (ms_per_step * 1e-3),
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "strong" if args.strong_total else "weak",
            "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": workload_config(world),
            "engine": {"kernel": kname,
                       "exchange": None if world == 1 else (
                           "fused NVLink peer stores in the fold kernel, protocol "
                           + os.environ.get("GPR_EXCHANGE", "default") if args.collective == "p2p" else "ncclAllGather"),
                       "timing": "K steps in one CUDA-event region after a device-side rendezvous of all ranks, "
                                 "max over ranks"},
            "per_step": per_step,
            "value_at_median_step": (samples_per_step / (per_step["median_us"] * 1e-6)
                                     if per_step.get("median_us") else None),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak,
                         "traffic": None if not traffic else traffic.get("dram_bytes_per_launch"),
                         "traffic_source": None if not traffic else
                         "STATIC record " + str(traffic.get("source")) + " — not re-measured by this run",
                         "peak_source": peak_src,
                         "kernel": "gpr::k_reduce_%s (one launch per step%s)" % (
                             kname, "; step time contains the bitmap exchange" if world > 1 else ""),
                         "algorithmic_bytes_per_launch": bytes_per_launch},
            "e2e": None if profiling_only else {"value": samples_per_step / e2e_s_per_step, "unit": UNIT,
                    "pod_decisions_per_sec": real_pods_total / e2e_s_per_step,
                    "ms_per_step": e2e_s_per_step * 1e3, "steps": e2e_steps,
                    "h2d_bytes_per_step": int(h_u.nbytes + h_e.nbytes),
                    "d2h_bytes_per_step": int(W_out * 4 + 24),
                    "api": "gpr_decide(ctx, window{mem_kind=HOST, pinned}, result{HOST})",
                    "bound": "PCIe (per rank)", "pcie": pcie,
                    "matches_device_path": e2e_ok},
            "single_decision_us": single_decision_us,
            "exchange_breakdown": breakdown,
            "e2e_resident": resident,
            "e2e_daemon_binary": daemon_binary,
            "e2e_u8": e2e_u8,
            "gpu_launches": int(launches), "clocks": clocks,
            "parity": "unchecked (--no-cpu)",
            "device": eng.device_info()["name"],
        }
        if not args.no_cpu and not profiling_only:
            # ---- the checker (the one place this arm runs the oracle; after every timed region) ----------
            chk = check_parity(world, first_bits, first_counts, last_bits, last_counts, last_window)
            ok = chk.pop("ok") and e2e_ok
            line["parity"] = "PASS" if ok else "FAIL"
            line["parity_detail"] = chk
            parity_failed = not ok
            if world == 1:
                line["cpu_baseline"] = cpu_baseline()
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 1 if parity_failed else 0


def check_parity(world, first_bits, first_counts, last_bits, last_counts, last_window):
    """rank 0: the gathered rank-major bitmap (== the global bitmap: shards are whole words) and the summed
    counts of two steps against the streaming CPU oracle over all world x PODS pods"""
    import numpy as np
    from oracle import oracle_c
    total = PODS * world
    n_words = (total + 31) // 32
    out = {"pods_checked": total, "steps_checked": ["pre-timing step (window 0)",
                                                    f"last timed step (window {last_window})"]}
    ok = True
    for name, win, bits, counts in (("first", 0, first_bits, first_counts),
                                    ("last", last_window, last_bits, last_counts)):
        ref = oracle_c.decide_synth(SEED + 16 * win, 0, total, GPUS, SAMPLES, use_elig=True)
        same_bits = bool(np.array_equal(bits[:n_words], ref["decision_bits"]) and not bits[n_words:].any())
        same_counts = list(counts) == [ref["n_series"], ref["n_candidates"], ref["n_decisions"]]
        out[name] = {"bitmap": same_bits, "counts": same_counts, "n_decisions": ref["n_decisions"]}
        ok = ok and same_bits and same_counts
    out["ok"] = ok
    return out


def cpu_baseline():
    """the oracle timed on this box's host cores over a bounded sample of the same workload"""
    from oracle import oracle_c
    n_threads = oracle_c.hardware_threads()
    run, dbits, counts = cpu_pass_factory(n_threads)
    run(0)
    t0 = time.perf_counter()
    run(1)
    one = time.perf_counter() - t0
    passes = max(4, min(2000, int(3.0 / max(one, 1e-4))))
    best = float("inf")
    for _ in range(4):               # best of 4 x ~3 s
        t0 = time.perf_counter()
        for i in range(passes):
            run(i)
        best = min(best, time.perf_counter() - t0)
    t1 = time.perf_counter()
    run(2, PODS, 1)
    one_thread = time.perf_counter() - t1
    samples = PODS * GPUS * SAMPLES
    return {"value": samples * passes / best, "unit": UNIT, "cores": n_threads, "kind": "port",
            "pod_decisions_per_sec": PODS * passes / best,
            "single_thread_value": samples / one_thread,
            "host_stream_gbs": samples * passes / best * 4 / 1e9,
            "sample": f"best of 4 x {passes} passes over {ROTATE} rotated C2 windows ({samples * 4 / 1e6:.0f} MB each, "
                      f"host RAM), {n_threads} pinned POSIX threads; oracle/gpr_oracle.c -O3 -march=x86-64-v3, scalar f64"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--kernel", default=os.environ.get("GPR_BENCH_KERNEL", "auto"),
                    choices=["auto", "ldg", "tma"])
    ap.add_argument("--e2e-steps", type=int, default=50)
    ap.add_argument("--collective", default="p2p", choices=["p2p", "nccl"],
                    help="N > 1: bitmap exchange fused into the kernel over peer memory, or one ncclAllGather")
    ap.add_argument("--no-cpu", action="store_true", help="skip the oracle legs (parity check, cpu_baseline)")
    ap.add_argument("--no-breakdown", action="store_true", help="N > 1: skip the exchange breakdown passes")
    ap.add_argument("--no-daemon-binary", action="store_true", help="skip the daemon-mode run of the gpu-pruner binary")
    ap.add_argument("--config", default="c2", choices=["c2", "c4", "c5"],
                    help="c2 (default, the judged workload): 10k pods x 4 x 1800 per GPU, weak scaling.  "
                         "c4 / c5 (profiling only): BASELINE configs[3] / [4], a FIXED total of 250k x 4 x 1800 "
                         "/ 2.5M x 4 x 7200 pods sharded over the ranks (strong scaling)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    global PODS, GPUS, SAMPLES, ROTATE
    args.strong_total = 0
    if args.config != "c2":
        world = int(os.environ.get("WORLD_SIZE", "1"))
        total, GPUS, SAMPLES = (250000, 4, 1800) if args.config == "c4" else (2500000, 4, 7200)
        args.strong_total = total
        PODS = total // world           # pods per rank (both totals divide by 1, 2, 4, 8)
        ROTATE = 2 if args.config == "c4" else 1
        args.no_cpu = True
        args.e2e_steps = min(args.e2e_steps, 3)
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)
    return run_cuda(args)


if __name__ == "__main__":
    sys.exit(main())
