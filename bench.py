#!/usr/bin/env python
"""bench.py -- PG-loss + CTC utterances/s on B200 (BASELINE.json metric), one JSON line on stdout.

    python bench.py --gpus N --steps K --warmup W            our CUDA path (one process per GPU under torchrun)
    python bench.py --impl reference --steps K --warmup W    the CPU arm: the oracle port on the host cores
    python bench.py --config {1,2,3,4} ...                   which BASELINE.json configs[] entry (default 1)
    python bench.py ... --dump-outputs DIR                   also write the last timed step's outputs as DIR/<name>.npy

configs[1] (default, the headline): a step is one pass of the hot path (sample K hypotheses -> collapse -> edit
distance -> reward -> baseline -> REINFORCE gradient, plus CTC alpha-beta loss and gradient; loss scalar + dlogits
out) over one batch of B synthetic utterances per GPU: B=64, T=500, V=30, K=16, label length 100.  Utterances are
independent, so N GPUs run N batches with no data-path collective (scaling: weak).
configs[2]: the CTC alpha-beta loss + gradient alone, B=128, T=1000, V=30, label length 200.
configs[3]: full PG training step (acoustic model fwd/bwd + fused PG loss + optimiser), global B=256 split over the
            N GPUs (scaling: strong), NCCL all-reduce of the model gradients (DDP); the all-reduce is also timed alone.
configs[4]: the stress grid K in {4,16,64} x T in {250,1000,2000} (label length up to 400), B=32 per GPU on every GPU,
            whole step + every stand-alone kernel with its GB/s.

The timed loop of configs[1]/[2] contains no Python per step: the steps are enqueued by pgasr_pg_ctc_step_multi
(functional.StepQueue), one C-ABI call per chunk of steps, outputs preallocated.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

L2_BYTES = 126 * 1024 * 1024
METRIC = "pg_ctc_loss_utterances_per_sec"
SHAPES = {1: dict(batch=64, T=500, V=30, K=16, L=100, w_pg=1.0, w_ctc=1.0),
          2: dict(batch=128, T=1000, V=30, K=16, L=200, w_pg=0.0, w_ctc=1.0)}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=1, choices=[1, 2, 3, 4], help="BASELINE.json configs[] index")
    ap.add_argument("--batch", type=int, default=0, help="utterances per GPU per step (0: the config's)")
    ap.add_argument("--T", type=int, default=0)
    ap.add_argument("--V", type=int, default=0)
    ap.add_argument("--K", type=int, default=0)
    ap.add_argument("--L", type=int, default=0)
    ap.add_argument("--regime", default="random", choices=["random", "peaky"])
    ap.add_argument("--reward", default="ed", choices=["ed", "cer", "ed_to_go"])
    ap.add_argument("--cpu-batch", type=int, default=0, help="utterances per CPU step (0: same as --batch)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--w-pg", type=float, default=None, help="diagnosis: override the PG weight (0 drops the PG role)")
    ap.add_argument("--w-ctc", type=float, default=None, help="diagnosis: override the CTC weight (0 drops the CTC role)")
    ap.add_argument("--python-loop", action="store_true", help="one functional.pg_ctc_step call per step (round-1 loop)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step (rank 0) as DIR/<name>.npy; configs[1] and [2]")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and (args.impl != "ours" or args.config not in (1, 2)):
        ap.error("--dump-outputs covers the GPU path of configs[1] and configs[2]")
    sh = SHAPES.get(args.config, SHAPES[1])
    for k in ("batch", "T", "V", "K", "L"):
        if not getattr(args, k):
            setattr(args, k, sh[k])
    w_pg, w_ctc = args.w_pg, args.w_ctc
    args.w_pg, args.w_ctc = sh["w_pg"], sh["w_ctc"]
    if w_pg is not None:
        args.w_pg = w_pg
    if w_ctc is not None:
        args.w_ctc = w_ctc
    return args


def algorithmic_bytes_per_utt(args):
    # SURVEY.md 8(d): read logits + write dlogits + targets + lengths + nll (+ R[K], logp[K] with the PG part)
    T, V, L, K = args.T, args.V, args.L, args.K
    return 8 * T * V + 4 * L + 8 * K + 12 if args.w_pg else 8 * T * V + 4 * L + 4


def algorithmic_ops(args, utt_per_s):
    """SURVEY.md 8(d): algorithmic op counts per utterance next to the byte roofline (the path is bound by serial depth
    and ALU work, not by bytes).  Hypothesis length: ~0.93 T for random logits, ~L for peaky ones (SURVEY's figures)."""
    T, V, K, L = args.T, args.V, args.K, args.L
    S = 2 * L + 1
    lh = int(round(0.93 * T)) if args.regime == "random" else L
    per = {}
    if args.w_pg:
        per.update({"sampler_exp": T * V, "sampler_cdf_compares_linear_scan": K * T * V, "sampler_draws": K * T,
                    "levenshtein_cells": K * lh * L, "levenshtein_dependent_diagonals": lh + L - 1})
    if args.w_ctc:
        per.update({"ctc_state_updates_alpha_plus_beta": 2 * T * S, "ctc_dependent_frames": T})
    rates = {k + "_per_s": v * utt_per_s for k, v in per.items() if "dependent" not in k}
    return {"per_utterance": per, "achieved": rates, "hyp_len_assumed": lh if args.w_pg else None}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


def traffic_from_profile(workload_key):
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            if d.get("workload") == workload_key:
                return d.get("dram_bytes_per_launch")
        except Exception:
            pass
    return None


def pool_size(args):
    bytes_logits = args.batch * args.T * args.V * 4
    return max(2, -(-int(1.25 * L2_BYTES) // bytes_logits)), bytes_logits      # rotating inputs: pool footprint > L2


DUMP_BYTES = 64 * 2**20


def dump_outputs(directory, outputs):
    """outputs: name -> torch tensor, as the step returned them.  Written as float32 (float64 stays float64, integers
    become float64, which holds them exactly).  Past DUMP_BYTES in all, an array over its share of the budget is
    replaced by the same seeded sample of its flattened elements on every run, so that two builds stay comparable."""
    arrays = {}
    for name, t in outputs.items():
        a = t.detach().cpu().numpy()
        arrays[name] = a if a.dtype in (np.float32, np.float64) else a.astype(np.float64)
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(directory, exist_ok=True)
    for name, a in sorted(arrays.items()):
        share = DUMP_BYTES // len(arrays) // a.itemsize
        if total > DUMP_BYTES and a.size > share:
            sys.stderr.write(f"dump-outputs: {name} is a seeded sample of {share} of its {a.size} elements\n")
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, share, replace=False))]
        np.save(os.path.join(directory, name + ".npy"), a)


def workload_config(args):
    B = args.batch
    pool, bytes_logits = pool_size(args)
    what = "PG loss (sample/collapse/edit-distance/reward/baseline/gradient) + CTC" if args.w_pg else \
        "CTC alpha-beta loss + gradient alone"
    return {"workload": f"configs[{args.config}]: {what}, B={B}/GPU, T={args.T}, V={args.V}, K={args.K}, "
                        f"label_len={args.L}, {args.regime} logits",
            "B_per_gpu": B, "T": args.T, "V": args.V, "K": args.K, "L": args.L, "regime": args.regime,
            "reward": args.reward, "baseline": "mean", "pg_weight": args.w_pg, "ctc_weight": args.w_ctc,
            "rng": "philox4x32-10",
            "l2": f"inputs (and outputs) rotate over a pool of {pool} distinct batches "
                  f"({pool * bytes_logits / 2**20:.0f} MiB of logits > 126 MiB L2)"}


# --------------------------------------------------------------------------------------------- CPU arm
def cpu_step_fn(args, B):
    from oracle import cport
    from tests.synth import make_batch
    cport.set_num_threads(os.cpu_count() or 1)          # torchrun exports OMP_NUM_THREADS=1; the CPU arm uses all cores
    logits, targets, in_len, tgt_len, _ = make_batch(B, args.T, args.V, args.K, args.L, seed=1234, regime=args.regime)
    kw = {"reward_mode": {"ed": 0, "cer": 1, "ed_to_go": 2}[args.reward]} if args.reward != "ed" else {}

    def step(i):
        return cport.pg_ctc_step(logits, targets, in_len, tgt_len, None, seed=0x5EED + i, K=args.K,
                                 w_pg=args.w_pg, w_ctc=args.w_ctc, **kw)
    return step, cport.max_threads()


def cpu_reference_leg(args, B=2):
    """The real upstream functions (metrics.edit_dist, CTCdecoder.collapse_fn copied verbatim into oracle/_ref by
    oracle/make_ref.py) around torch-CPU for the parts upstream has no code for -- BASELINE.md section 3."""
    try:
        from oracle import refpath
        if not refpath.available():
            return None
        return refpath.time_step(B, args.T, args.V, args.K, args.L, regime=args.regime, w_pg=args.w_pg, w_ctc=args.w_ctc)
    except Exception as e:                               # the leg is informational; never fail the bench on it
        return {"error": repr(e)[:200]}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    if args.config in (3, 4):
        emit({"impl": "reference", "unavailable": f"configs[{args.config}] has no CPU arm (the acoustic model and the "
              "stress grid are measured on the GPU only); the CPU arm covers configs[1] and configs[2]"})
        return 0
    B = args.cpu_batch or args.batch
    step, cores = cpu_step_fn(args, B)
    for i in range(args.warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(i)
    dt = time.perf_counter() - t0
    val = B * args.steps / dt
    sample = (f"{args.steps} steps x {B} utterances (T={args.T},V={args.V},K={args.K},L={args.L}), C oracle port, "
              "OpenMP over utterances")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "utt/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(args.steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args),
        "note": "CPU arm; upstream is pure Python, so this is the C port of it (far faster than upstream's loops)",
        "cpu_baseline": {"value": val, "unit": "utt/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "utt/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    ref = cpu_reference_leg(args)
    if ref:
        line["cpu_baseline_reference"] = ref
    emit(line)
    return 0


# --------------------------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    """Polls NVML for SM clock and throttle reasons while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def sample(self):
        if not self.ok:
            return
        nv = self.nv
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
                     0x80: "hw_power_brake_slowdown"}
            for bit, nm in names.items():
                if r & bit:
                    self.reasons.add(nm)
        except Exception:
            pass

    def run(self):
        while not self.stop_flag:
            self.sample()
            time.sleep(0.002)

    def result(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# --------------------------------------------------------------------------------------------- GPU arm
class Dist:
    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise RuntimeError("bench.py (impl ours) needs a CUDA device; there is no CPU fallback")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.solo = bool(os.environ.get("PGASR_BENCH_NO_DIST"))      # diagnosis only: ranks run unsynchronised, rank 0 reports itself
        if self.world > 1 and not self.solo:
            dist.init_process_group("nccl", device_id=self.dev)
        from pgasr_b200 import _native
        if not os.path.exists(_native.LIB_PATH):             # the library normally travels with the snapshot; else build it here
            if self.rank == 0:
                import __graft_entry__
                __graft_entry__.build()
            if self.world > 1:
                dist.barrier()
        assert _native.lib().pgasr_device_check() == 0, "not an sm_100 device"

    def barrier(self):
        if self.world > 1 and not self.solo:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if self.world > 1 and not self.solo:
            t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            return float(t[0])
        return x

    def close(self):
        if self.world > 1 and not self.solo:
            self.dist.destroy_process_group()


def run_ours(args):
    import torch
    import pgasr_b200
    from pgasr_b200 import _native, functional as F
    from tests.synth import make_batch

    D = Dist()
    world, rank, dev = D.world, D.rank, D.dev
    B, T, V, K, L = args.batch, args.T, args.V, args.K, args.L
    pool, bytes_logits = pool_size(args)
    host, devb = [], []
    for i in range(pool):
        lg, tg, il, tl, _ = make_batch(B, T, V, K, L, seed=1000 * rank + i, regime=args.regime)
        h = {"logits": torch.from_numpy(lg).pin_memory(), "targets": torch.from_numpy(tg).pin_memory(),
             "in_len": torch.from_numpy(il).pin_memory(), "tgt_len": torch.from_numpy(tl).pin_memory()}
        host.append(h)
        devb.append({k: v.to(dev) for k, v in h.items()})
    # every output buffer is allocated here, once; the timed loop is one C-ABI call per chunk of <= pool steps
    queue = F.StepQueue(devb, K=K, reward=args.reward, pg_weight=args.w_pg, ctc_weight=args.w_ctc,
                        want=("rewards", "nll") if args.w_pg else ("nll",))

    def run_steps(first, n):
        """Steps first .. first + n - 1 (batch i % pool, seed 0x5EED + i); returns the outputs of the last one."""
        if args.python_loop:
            for i in range(first, first + n):
                b = devb[i % pool]
                out = F.pg_ctc_step(b["logits"], b["targets"], b["in_len"], b["tgt_len"], K=K, seed=0x5EED + i,
                                    reward=args.reward, pg_weight=args.w_pg, ctc_weight=args.w_ctc,
                                    workspace=queue.workspace, want=("rewards", "nll") if args.w_pg else ("nll",))
            return {k: v for k, v in out.items() if isinstance(v, torch.Tensor)}
        done = 0
        while done < n:
            c = min(pool, n - done)
            queue.run(first=first + done, n=c, seed=0x5EED + first + done)
            done += c
        return queue.outputs[(first + n - 1) % pool]

    # ---- device-resident throughput ("value") --------------------------------------------------
    # warm-up: at least W (>= 3) steps, and at least ~30 ms of them so that the SM clock has left its idle state before
    # the timed region (a 20-step run is 1 ms of GPU time; the clocks line of the JSON shows what the timed region saw).
    # The clock-driven part repeats steps first .. first + pool - 1, so the timed steps start at step `first` however
    # long it ran: their batches and seeds, and so their outputs, depend on the arguments alone.
    first = warm = max(args.warmup, 3)
    run_steps(0, warm)
    torch.cuda.synchronize()
    t_w = time.perf_counter()
    while time.perf_counter() - t_w < 0.03:
        run_steps(first, pool)
        torch.cuda.synchronize()
        warm += pool
    D.barrier()
    sampler = ClockSampler(D.local)
    sampler.start()
    launches0 = _native.lib().pgasr_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    last = run_steps(first, args.steps)
    e1.record()
    sampler.sample()
    torch.cuda.synchronize()
    sampler.sample()
    ms = D.max_over_ranks(e0.elapsed_time(e1))
    launches = _native.lib().pgasr_launch_count() - launches0
    if args.dump_outputs and rank == 0:                  # before the steps below overwrite the queue's outputs
        dump_outputs(args.dump_outputs, last)
    D.barrier()
    sampler.stop_flag = True
    sampler.join(1.0)
    value = world * B * args.steps / (ms * 1e-3)

    # ---- dominant kernel (roofline): the step IS one launch of pg_ctc_fused_kernel, so its average launch duration
    # over the timed region is that region's CUDA-event time / launches -- the same clock as `value` (back-to-back
    # launches overlap their heads and tails under programmatic dependent launch; bracketing every launch with its
    # own event pair would break that overlap and time a different thing).  The isolated figure is reported beside it.
    nrep = min(args.steps, 50)
    pairs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(nrep)]
    for i, (k0, k1) in enumerate(pairs):
        k0.record()
        queue.run(first=i, n=1, seed=i)
        k1.record()
    torch.cuda.synchronize()
    isolated_ms = sum(k0.elapsed_time(k1) for k0, k1 in pairs) / nrep
    per_step_launches = launches / max(args.steps, 1)
    kernel_ms = ms / max(launches, 1)
    peak, peak_src = measured_peak()
    step_bytes = B * algorithmic_bytes_per_utt(args)             # SURVEY.md 8(d): 120 540 B/utt at the headline shape
    achieved = step_bytes / (kernel_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm",
                "kernel": "pg_ctc_fused_kernel (the whole step: 1 launch)" if per_step_launches == 1 else
                          f"{per_step_launches:g} launches per step",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "peak_source": peak_src + " (MEASURED_PEAKS.json hbm_gbs, burst copy)" if peak_src == "measured" else peak_src,
                "traffic": traffic_from_profile(f"B={B},T={T},V={V},K={K},L={L}"),
                "algorithmic_bytes_per_launch": step_bytes, "kernel_ms": kernel_ms,
                "kernel_ms_isolated": isolated_ms, "launches_per_step": per_step_launches,
                "note": "latency bound, not bandwidth bound: T dependent lattice frames per utterance and only "
                        f"2B={2 * B} CTAs of work; see DESIGN.md section 5"}

    # ---- end to end through the public host-buffer API ("e2e"): pinned HOST inputs and outputs, every step copies
    # its logits/targets/lengths H2D and its loss, rewards, nll AND the full dlogits D2H inside the timed region;
    # HostPipeline keeps `depth` steps in flight so the copies of neighbouring steps overlap the kernel ----------
    e2e = None
    if not args.no_e2e:
        depth = 4
        pipe = pgasr_b200.HostPipeline(B, T, V, K, L, depth=depth, reward=args.reward, pg_weight=args.w_pg,
                                       ctc_weight=args.w_ctc)
        outs = [pipe.output_buffers() for _ in range(depth)]

        def e2e_step(i):
            h = host[i % pool]
            return pipe.submit(h["logits"], h["targets"], h["in_len"], h["tgt_len"], out=outs[i % depth], seed=0x5EED + i)
        for i in range(warm):
            e2e_step(i)
        pipe.wait()
        D.barrier()
        t0 = time.perf_counter()
        for i in range(args.steps):
            e2e_step(i)
        pipe.wait()
        torch.cuda.synchronize()
        dt = D.max_over_ranks(time.perf_counter() - t0)
        # single-step latency (submit + wait, nothing else in flight)
        lat = []
        for i in range(20):
            t1 = time.perf_counter()
            pipe.wait(e2e_step(i))
            lat.append(time.perf_counter() - t1)
        pipe.close()
        h2d = bytes_logits + B * L * 4 + 2 * B * 4
        d2h = bytes_logits + (B * K + B + 4) * 4
        e2e = {"value": world * B * args.steps / dt, "unit": "utt/s", "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "ms_per_step": 1e3 * dt / args.steps,
               "api": f"HostPipeline.submit/wait (pgasr_host_* C ABI), depth {depth}, pinned host buffers",
               "outputs_to_host": "loss, rewards[B,K], nll[B], dlogits[B,T,V]",
               "sync_step_latency_ms": 1e3 * statistics.median(lat)}

    # ---- CPU baseline on rank 0 at N=1 ----------------------------------------------------------------
    cpu = cpu_ref = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        Bc = args.cpu_batch or B
        cstep, cores = cpu_step_fn(args, Bc)
        t0 = time.perf_counter()
        cstep(0)
        first = time.perf_counter() - t0
        reps = int(min(max(round(10.0 / max(first, 1e-3)), 1), 20))
        t0 = time.perf_counter()
        for i in range(reps):
            cstep(i + 1)
        dt = time.perf_counter() - t0
        cpu = {"value": Bc * reps / dt, "unit": "utt/s", "cores": cores, "kind": "port",
               "sample": f"{reps} steps x {Bc} utterances of the same workload, C oracle port (OpenMP over utterances)"}
        cpu_ref = cpu_reference_leg(args)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "utt/s", "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 I/O and sampler, f64 CTC lattice, integer collapse/edit distance", "data": "synthetic",
            "config": workload_config(args),
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches),
            "clocks": sampler.result(),
            "launch_path": "functional.pg_ctc_step per step (Python)" if args.python_loop else
                           f"pgasr_pg_ctc_step_multi: one C-ABI call per {min(pool, args.steps)} steps; consecutive steps of a "
                           "call overlap on three streams (independent batches, own workspace lane each)",
        }
        if cpu_ref:
            line["cpu_baseline_reference"] = cpu_ref
        try:
            line["algorithmic_ops"] = algorithmic_ops(args, value)
        except Exception:                                   # (reporting only: never in the way of the line)
            pass
        emit(line)
    D.close()
    return 0


# --------------------------------------------------------------------------------------------- configs[3]
def run_config3(args):
    """Full PG training step, data parallel, global batch 256 (strong scaling); see examples/acoustic_harness.py."""
    sys.path.insert(0, os.path.join(ROOT, "examples"))
    import acoustic_harness
    D = Dist()
    res = acoustic_harness.run(D, global_batch=256 if not args.batch or args.batch == 64 else args.batch * D.world,
                               T=args.T, V=args.V, K=args.K, L=args.L, steps=args.steps, warmup=max(args.warmup, 3))
    if D.rank == 0:
        line = {"metric": METRIC, "value": res["utt_per_s"], "unit": "utt/s", "n_gpus": D.world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": res["ms_per_step"], "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f32 (cuDNN BLSTM f32, loss as configs[1])",
                "data": "synthetic",
                "config": {"workload": f"configs[3]: full PG training step (acoustic model fwd/bwd + fused PG+CTC loss + Adam), "
                                       f"global B={res['global_batch']}, T={args.T}, V={args.V}, K={args.K}, label_len={args.L}, "
                                       f"DDP over {D.world} GPU(s)", "global_batch": res["global_batch"],
                           "B_per_gpu": res["B_per_gpu"], "T": args.T, "V": args.V, "K": args.K, "L": args.L,
                           "l2": "activations of the 3-layer BLSTM per step exceed the L2"},
                "breakdown": res, "roofline": None, "cpu_baseline": None, "e2e": None,
                "gpu_launches": res.get("loss_launches_per_step", 1) * args.steps}
        emit(line)
    D.close()
    return 0


# --------------------------------------------------------------------------------------------- configs[4]
def run_config4(args):
    """Stress grid on every GPU: whole step + stand-alone kernels, ms = max over ranks."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import sweep
    D = Dist()
    B = args.batch if args.batch != 64 else 32
    cases, tot_utt, tot_ms = [], 0, 0.0
    for K in (4, 16, 64):
        for T, L in ((250, 50), (1000, 200), (2000, 400)):
            c = sweep.case(B, T, 30, K, L, dev=D.dev, seed=1000 * D.rank + T + K, reps=max(args.steps // 20, 5), quiet=True)
            for name, k in c["kernels"].items():
                k["ms"] = D.max_over_ranks(k["ms"])
                k["algorithmic_GBps"] = round(k["bytes"] / k["ms"] / 1e6, 2)
            step_ms = c["kernels"]["whole step (pgasr_pg_ctc_step)"]["ms"]
            c["step_utt_per_s"] = round(D.world * B / step_ms * 1e3, 1)
            tot_utt += D.world * B
            tot_ms += step_ms
            cases.append(c)
    if D.rank == 0:
        sweep.merge_measured_traffic(cases, os.path.join(ROOT, "profiles", "r02_sweep_ncu.jsonl"))
        line = {"metric": METRIC, "value": tot_utt / (tot_ms * 1e-3), "unit": "utt/s", "n_gpus": D.world,
                "steps": len(cases), "warmup": 3, "ms_per_step": tot_ms / len(cases), "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32 / f64 lattice / integer", "data": "synthetic",
                "config": {"workload": f"configs[4]: stress grid K in {{4,16,64}} x (T,L) in {{(250,50),(1000,200),(2000,400)}}, "
                                       f"V=30, B={B}/GPU on each of {D.world} GPU(s); value = utterances of one pass over the "
                                       "grid / summed step times", "B_per_gpu": B,
                           "l2": "each shape is timed alone over 20+ repetitions of one batch (L2 resident inputs for the "
                                 "small shapes: the kernels are latency bound, see DESIGN.md)"},
                "cases": cases, "roofline": None, "cpu_baseline": None, "e2e": None, "gpu_launches": None}
        emit(line)
    D.close()
    return 0


_JSON_FD = None


def emit(line):
    """The one JSON line goes to the process's ORIGINAL stdout; see main()."""
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    global _JSON_FD
    args = parse()
    # stdout must carry exactly one JSON line: libraries that print there (NCCL's version banner under torchrun) are
    # sent to stderr by pointing fd 1 at fd 2 for the lifetime of the run; the JSON line is written to the saved fd
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference(args)
    if args.config == 3:
        return run_config3(args)
    if args.config == 4:
        return run_config4(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
