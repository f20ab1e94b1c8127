#!/usr/bin/env python
"""Benchmark of the fused D3PM reverse-diffusion token update (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

`--steps` sets the timed steps of the headline metric.  `--dump-outputs DIR` (`--impl ours` only) writes the tokens of
the last timed step to DIR/x_prev.npy.

A "step" is ONE fused reverse step (classifier-free guidance + posterior + Gumbel-max sample, production
in-kernel Philox mode) over one batch of synthetic logits.  Workload at N GPUs: BASELINE config 2 per GPU
(16 videos x 16x16x16 token grid x 4096 codes + [MASK], guidance 2, t = 50) — the batch of videos is
partitioned across ranks with no data-path collective (weak scaling: 16 videos per GPU, which at 8 GPUs
is exactly config 4's B = 128).  Prints ONE JSON line on rank 0.

  value      token updates / s with the logits already resident in HBM (whole job, all ranks)
  e2e        the same through the host-buffer C entry `d3pm_host_step_run` (`ops.HostStep`) with pinned HOST logits:
             H2D + kernel + D2H every step; per-rank H2D GB/s and CPU affinity are reported next to it
  roofline   algorithmic bytes (32 784 B / token update, BASELINE.md §3) / kernel time vs the measured HBM peak
  cpu_baseline  the reference's own `p_sample` (unmodified module, staged under baseline/_ref) on the host cores, on a
             bounded sample of the batch, rank 0 only (the oracle port only where no copy of the reference is present)
  sustained  the same step, 1500 back to back (power-capped regime)
  config4_gather_check  (N > 1) the token all-gather timed, and rank 0's recomputation of other ranks' videos: bit-identical
  configs    config 4 as written (128 videos split over the ranks, strong scaling) and config 5 (64 videos, guidance on/off)
  next_rows  config 3 with the reference's real denoiser (reference sample loop on the GPU vs the drop-in, same weights),
             fused head, training loss + gradient, purity prior, q_sample, the host entry of the fused head

`--impl reference` times the reference's own `p_sample` alone on the host cores at the full config-2 batch (16 videos per
step) - the same `config` as our arm.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

T_STEPS, K_CODES, GRID = 100, 4096, (16, 16, 16)
N_TOKENS = GRID[0] * GRID[1] * GRID[2]
VIDEOS_PER_GPU = 16
GUIDANCE, T_NOW = 2.0, 50
BYTES_PER_TOKEN = 2 * K_CODES * 4 + 8 + 8  # both logit rows + x_t + x_{t-1}
METRIC, UNIT = "reverse_step_token_updates_per_sec", "token-updates/s"


def workload_name(n_gpus, videos_per_gpu=VIDEOS_PER_GPU):
    return (f"config2 x{n_gpus}: {videos_per_gpu} videos/GPU, 16x16x16 grid, {K_CODES}+1 classes, guidance {GUIDANCE:g}, "
            f"t={T_NOW}, fp32 logits, in-kernel Philox Gumbel-max")


def config_dict(world, videos_per_gpu=VIDEOS_PER_GPU):
    """The `config` object of the JSON line: the same for our arm and for `--impl reference`."""
    return {"workload": workload_name(world, videos_per_gpu), "global_batch": videos_per_gpu * world, "tokens_per_video": N_TOKENS,
            "classes": K_CODES + 1,
            "cache": f"inputs {videos_per_gpu * N_TOKENS * BYTES_PER_TOKEN / 1e9:.2f} GB per GPU >> 126 MB L2, re-read every step (no flush needed)",
            "parallelism": f"batch of videos partitioned over {world} GPU(s), no collective in the step"}


# ----------------------------------------------------------------------------- CPU reference arm
def _host_ram_gb():
    try:
        import psutil
        return psutil.virtual_memory().available / 1e9
    except Exception:
        return 0.0


def cpu_reference(steps, warmup, sample_videos=VIDEOS_PER_GPU):
    """Time the reference's OWN `p_sample` (diffusion_transformer.py:304-352, unmodified module from
    `baseline/reference_loader.py`: /root/reference here, the staged baseline/_ref on the GPU box) on the host cores, on
    `sample_videos` videos of the workload per step; its denoiser is a stub that hands back pre-generated logits the way
    `Text2ImageTransformer` does (a [B, K, N] view of [B, N, K]), so only the update is timed, as on the GPU arm.
    Falls back to the oracle port (bit-for-bit pinned to the reference by tests/golden) only when no copy of the
    reference is present, and says so in `kind`."""
    import torch

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    B, N, K = sample_videos, N_TOKENS, K_CODES
    g = torch.Generator().manual_seed(0)
    lc = torch.randn(B, N, K, generator=g)
    lu = torch.randn(B, N, K, generator=g)
    t = torch.full((B,), T_NOW, dtype=torch.int64)

    from baseline import reference_loader as RL
    if RL.reference_available():
        kind = "reference"

        class Stub(torch.nn.Module):  # the three attributes DiffusionTransformer touches + the denoiser's output layout
            def __init__(self):
                super().__init__()
                self.content_emb = type("E", (), {"num_embed": K + 1})()
                self.to_logits = torch.nn.Sequential(torch.nn.Identity(), torch.nn.Linear(1, 1))

            def forward(self, x_t, cond, t_):
                return (lc if float(cond.flatten()[0]) > 0.5 else lu).permute(0, 2, 1)

        model = RL.build_reference_model(Stub(), diffusion_step=T_STEPS, guidance_scale=GUIDANCE, content_seq_len=N)
        p_mask = float(model.log_cumprod_ct[T_NOW].exp())
        x_t = torch.where(torch.rand(B, N, generator=g) < p_mask, torch.full((B, N), K), torch.randint(0, K, (B, N), generator=g))
        log_x_t = RL.load_diffusion_module().index_to_log_onehot(x_t, K + 1)
        cond, cf = torch.ones(B, 1, 1), torch.zeros(B, 1, 1)

        def step():
            model.p_sample(log_x_t, cond, cf, t, [0] * B, model.n_sample[T_NOW])
    else:
        kind = "port"
        from oracle import d3pm_oracle as O
        sched = O.make_schedule(T_STEPS, K)
        p_mask = float(sched["log_cumprod_ct"][T_NOW].exp())
        x_t = torch.where(torch.rand(B, N, generator=g) < p_mask, torch.full((B, N), K), torch.randint(0, K, (B, N), generator=g))
        log_x_t = O.index_to_log_onehot(x_t, K + 1)
        u = torch.rand(B, K + 1, N, generator=g)
        lc_l, lu_l = lc.permute(0, 2, 1), lu.permute(0, 2, 1)

        def step():
            O.p_sample_step(sched, lc_l, lu_l, log_x_t, t, GUIDANCE, u)

    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            step()
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    per_step = sum(times) / len(times)
    tokens = B * N
    what = ("the reference's own DiffusionTransformer.p_sample (unmodified module)" if kind == "reference"
            else "oracle port of p_sample (no copy of the reference on this box)")
    return {"value": tokens / per_step, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": f"{what}: {B} video(s) x {N} tokens x {K + 1} classes per step, {len(times)} timed step(s) after {warmup} "
                      f"warm-up, {per_step * 1e3:.0f} ms/step, torch {torch.__version__} CPU, {cores} threads"}, per_step


def run_reference(args):
    """`--impl reference`: the reference's CPU implementation of the path on this box's host cores, on OUR arm's config
    (config 2: 16 videos per step) whenever the host has the memory for it (peak ~25 GB of fp32/fp64 temporaries).
    `--steps` / `--warmup` are honoured up to 20 / 5 (a 16-video step takes ~7 s on 16 cores: the run ends within minutes)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ram = _host_ram_gb()
    videos = VIDEOS_PER_GPU if ram >= 48 else (4 if ram >= 16 else 1)
    steps, warmup = max(1, min(args.steps, 20)), max(1, min(args.warmup, 5))
    base, per_step = cpu_reference(steps, warmup, sample_videos=videos)
    note = (f"each step is the full config-2 batch ({videos} videos)" if videos == VIDEOS_PER_GPU else
            f"each step is a {videos}-video sample of the 16-video batch (host RAM available {ram:.0f} GB)")
    base["sample"] += (f"; {note}; rank 0 only (the CPU path does not use the GPUs; its throughput per step does not depend on how "
                       f"many such batches the job holds)")
    line = {
        "impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": per_step * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(args.gpus),
        "cpu_baseline": base,
        "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    """Polls NVML (SM clock, throttle reasons, power) for one device while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as exc:  # NVML missing: report it, do not invent clocks
            self.err = repr(exc)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        while not self.stop_flag.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                power = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                self.samples.append((sm, reasons, power))
            except Exception:
                pass
            time.sleep(0.0005)

    def summary(self):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml_unavailable"]}
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        sms = sorted(s[0] for s in self.samples)
        seen = set()
        for _, r, _ in self.samples:
            for bit, name in names.items():
                if r & bit:
                    seen.add(name)
        return {"sm_mhz": sms[len(sms) // 2] if sms else None, "sm_max_mhz": self.max_sm, "reasons": sorted(seen),
                "samples": len(sms), "power_w_max": max((s[2] for s in self.samples), default=None)}


# ----------------------------------------------------------------------------- our arm
def _pin_to_gpu_numa_node(local_rank):
    """Bind this rank's host threads to the CPUs next to its GPU (NVML's ideal affinity) BEFORE any pinned host buffer is
    allocated, so that first-touch places the e2e staging memory on the GPU's NUMA node.  -> description for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        before = len(os.sched_getaffinity(0))
        pynvml.nvmlDeviceSetCpuAffinity(h)
        cpus = sorted(os.sched_getaffinity(0))
        return {"cpus": f"{cpus[0]}-{cpus[-1]}" if cpus else "", "n_cpus": len(cpus), "n_cpus_before": before}
    except Exception as exc:
        return {"error": repr(exc)}


def _video_inputs(b_global, N, K, p_mask, dev):
    """Synthetic inputs of ONE video, keyed by its GLOBAL index (any rank generates the same bits for the same video)."""
    import torch
    gen = torch.Generator(device=dev).manual_seed(1000 + b_global)
    lc = torch.randn(N, K, device=dev, generator=gen)
    lu = torch.randn(N, K, device=dev, generator=gen)
    x = torch.where(torch.rand(N, device=dev, generator=gen) < p_mask, torch.full((N,), K, device=dev),
                    torch.randint(0, K, (N,), device=dev, generator=gen))
    return lc, lu, x


def run_ours(args):
    import torch
    import torch.distributed as dist

    import d3pm_b200
    from d3pm_b200 import _lib, ops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run for N>1")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    affinity = _pin_to_gpu_numa_node(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    # default: weak scaling, config 2 per GPU.  --global-videos G (config 4: G = 128): the SAME G videos split over the
    # ranks (strong scaling), G divisible by the world size
    if args.global_videos:
        if args.global_videos % world:
            raise SystemExit(f"--global-videos {args.global_videos} is not divisible by {world} ranks")
        B = args.global_videos // world
    else:
        B = VIDEOS_PER_GPU
    N, K = N_TOKENS, K_CODES
    B_global = B * world
    b0, b1 = d3pm_b200.shard_range(B_global, world, rank)
    row_offset = b0 * N

    # schedule + coefficient table from the module's own buffers (the product path, no oracle here)
    class _Stub(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.content_emb = type("E", (), {"num_embed": K + 1})()

    model = d3pm_b200.FusedDiffusionTransformer(transformer=_Stub(), diffusion_step=T_STEPS, alpha_init_type="alpha1",
                                                guidance_scale=GUIDANCE, content_seq_len=N).to(dev)
    table = model.coef_table()

    # synthetic inputs: N(0,1) logits, x_t masked with the schedule's probability at t; every video is generated from ITS
    # GLOBAL index, so a rank's shard is a slice of the one global batch whatever the world size (config 4's premise)
    p_mask = float(model.log_cumprod_ct[T_NOW].exp())
    logits_c = torch.empty(B, N, K, device=dev)
    logits_u = torch.empty(B, N, K, device=dev)
    x_t = torch.empty(B, N, dtype=torch.int64, device=dev)
    for i in range(B):
        logits_c[i], logits_u[i], x_t[i] = _video_inputs(b0 + i, N, K, p_mask, dev)
    t = torch.full((B,), T_NOW, dtype=torch.int64, device=dev)
    x_prev = torch.empty_like(x_t)
    status = ops.new_status(dev)
    launches = {"n": 0}

    def step(i):
        ops.fused_step(logits_c, logits_u, x_t, t, table, guidance_scale=GUIDANCE, sample_mode=_lib.SAMPLE_PHILOX,
                       seed=2024, offset=i, row_offset=row_offset, x_prev_out=x_prev, status=status)
        launches["n"] += 1

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for i in range(args.warmup):
        step(i)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches["n"] = 0
    ev0.record()
    for i in range(args.steps):
        step(args.warmup + i)
    ev1.record()
    barrier()
    timed_launches = launches["n"]
    sampler.stop_flag.set()
    sampler.join()
    elapsed_ms = ev0.elapsed_time(ev1)
    assert int(status.item()) & (_lib.STATUS_BAD_T | _lib.STATUS_BAD_TOKEN) == 0
    assert int(x_prev.min()) >= 0 and int(x_prev.max()) <= K
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, x_prev, B_global, rank)

    # ---- config 4's claim on hardware: the gathered tokens of the sharded job equal what ONE GPU computes for the same
    # global videos.  One step at a fixed offset on every rank, the (timed) token all-gather, then rank 0 regenerates
    # videos owned by OTHER ranks from their global seeds, runs them alone with their global row offset, and compares.
    gather = None
    if world > 1:
        step(4242)
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        gathered = d3pm_b200.gather_tokens(x_prev, B_global)  # warm-up of the communicator
        barrier()
        reps = 20
        g0.record()
        for _ in range(reps):
            gathered = d3pm_b200.gather_tokens(x_prev, B_global)
        g1.record()
        barrier()
        assert gathered.shape == (B_global, N)
        gather_us = g0.elapsed_time(g1) / reps * 1e3
        checked, mismatches = [], 0
        if rank == 0:
            for bg in sorted({B_global - 1, B, B_global // 2}):  # first video of rank 1, one in the middle, the very last
                lc1, lu1, x1 = _video_inputs(bg, N, K, p_mask, dev)
                one = ops.fused_step(lc1.unsqueeze(0), lu1.unsqueeze(0), x1.unsqueeze(0), t[:1], table, guidance_scale=GUIDANCE,
                                     sample_mode=_lib.SAMPLE_PHILOX, seed=2024, offset=4242, row_offset=bg * N)["x_prev"][0]
                mismatches += int((one != gathered[bg]).sum())
                checked.append(bg)
            assert mismatches == 0, f"sharded result differs from the single-GPU result on {mismatches} tokens"
        gather = {"all_gather_us": gather_us, "bytes_per_rank": B * N * 8, "collective": "all_gather_into_tensor (NCCL), int64 [B_local, N]",
                  "timed_reps": reps, "recomputed_on_rank0_global_videos": checked, "token_mismatches": mismatches,
                  "what": "one step on every rank, token all-gather timed on the device; rank 0 re-runs videos of other ranks from "
                          "their global seeds with their global row offset: bit-identical"}

    # ---- end to end through the host-buffer C entry (d3pm_host_step_run): pinned host logits, copies inside the timed region
    host = ops.HostStep(B, N, K, table, guidance=True, T=T_STEPS)
    h_c, h_u = logits_c.cpu().pin_memory(), logits_u.cpu().pin_memory()
    h_x, h_t = x_t.cpu().pin_memory(), t.cpu().pin_memory()
    e2e_steps = max(3, min(args.steps, 10))
    for i in range(2):
        host(h_c, h_u, h_x, h_t, guidance_scale=GUIDANCE, seed=2024, offset=i, row_offset=row_offset)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(e2e_steps):
        host(h_c, h_u, h_x, h_t, guidance_scale=GUIDANCE, seed=2024, offset=100 + i, row_offset=row_offset)
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    h2d_bytes, d2h_bytes = host.h2d_bytes, host.d2h_bytes
    host.close()
    del h_c, h_u

    # ---- the same step under sustained load (informational): after ~70 ms of back-to-back launches the board reaches its
    # power limit (NVML: sw_power_cap) and lowers the SM clock; a pure read of the same bytes does not
    sustained = None
    if world == 1:
        sus_steps = 1500
        barrier()
        sampler2 = ClockSampler(local_rank)
        sampler2.start()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for i in range(sus_steps):
            step(10_000 + i)
        s1.record()
        barrier()
        sampler2.stop_flag.set()
        sampler2.join()
        sus_ms = s0.elapsed_time(s1) / sus_steps
        sustained = {"steps": sus_steps, "ms_per_step": sus_ms, "value": B * N / (sus_ms * 1e-3), "unit": UNIT,
                     "GBps": B * N * BYTES_PER_TOKEN / (sus_ms * 1e-3) / 1e9, "clocks": sampler2.summary()}

    # ---- beyond the bench line (informational; the metric above is untouched): the other BASELINE configs and the rows
    # SURVEY §8 marks "next"
    extras, configs = {}, {}
    if not args.global_videos:
        try:
            time.sleep(1.0)
            del logits_c, logits_u
            torch.cuda.empty_cache()
            configs["config4_strong"] = measure_config4_strong(dev, model, table, world, rank, barrier)
            if world == 1:
                configs["config5"] = measure_config5(dev, model, table)
                configs["k2048"] = measure_k2048(dev)
                configs["logits_16bit"] = measure_16bit(dev, model, table)
        except Exception as exc:  # reported in the JSON line, never swallowed
            configs["error"] = repr(exc)
    if rank == 0 and world == 1:
        try:
            time.sleep(2.0)  # let the power controller settle after the sustained block
            global _NEXT_ROWS_LOGITS
            gen = torch.Generator(device=dev).manual_seed(1000)
            _NEXT_ROWS_LOGITS = (torch.randn(B, N, K, device=dev, generator=gen), torch.randn(B, N, K, device=dev, generator=gen))
            extras = measure_next_rows(dev, model, table, x_t, t, x_prev)
            _NEXT_ROWS_LOGITS = None
            torch.cuda.empty_cache()
            extras["decode"] = measure_decode(dev)
            extras["config3"] = measure_config3(dev)
        except Exception as exc:
            extras["error"] = repr(exc)

    times = torch.tensor([elapsed_ms, e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)  # max over ranks, measured on the device
    per_rank_e2e = [e2e_ms]
    if world > 1:
        every = [None] * world
        dist.all_gather_object(every, (e2e_ms, affinity))
        per_rank_e2e = [e[0] for e in every]
        affinity = [e[1] for e in every]
    elapsed_ms, e2e_ms = float(times[0]), float(times[1])

    if rank == 0:
        ms_per_step = elapsed_ms / args.steps
        tokens_global = B_global * N
        value = tokens_global / (ms_per_step * 1e-3)
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.isfile(peaks_path):
            peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
        else:
            peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
        achieved = B * N * BYTES_PER_TOKEN / (ms_per_step * 1e-3) / 1e9  # per GPU: one launch per step per rank
        traffic, traffic_src = None, None  # dram bytes per launch of the same kernel/workload, from the committed ncu capture
        for name in ("r02_summary.json", "r01_summary.json"):
            summ = os.path.join(ROOT, "profiles", name)
            if os.path.isfile(summ):
                sj = json.load(open(summ))
                traffic, traffic_src = sj.get("traffic_bytes_per_launch"), sj.get("source")
                break
        cpu_base, _ = cpu_reference(steps=2, warmup=1, sample_videos=4) if world == 1 else (None, None)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong" if args.global_videos else "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": config_dict(world, B),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "kernel": "step_stream_kernel<4, 8, true, false> (one launch per step)",
                         "algorithmic_bytes_per_launch": B * N * BYTES_PER_TOKEN,
                         "frac_of_nominal_8TBs": achieved / 8000.0},
            "e2e": {"value": tokens_global / (e2e_ms / e2e_steps * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                    "ms_per_step": e2e_ms / e2e_steps, "steps": e2e_steps,
                    "h2d_GBps_per_rank": [h2d_bytes / (m / e2e_steps * 1e-3) / 1e9 for m in per_rank_e2e],
                    "cpu_affinity_per_rank": affinity,
                    "api": "C ABI d3pm_host_step_run via d3pm_b200.ops.HostStep (pinned host logits -> chunked H2D overlapped with "
                           "d3pm_fused_step -> host tokens); the step is 2.15 GB of fp32 logits per rank on PCIe, see e2e of the "
                           "hidden-state entry in next_rows"},
            "gpu_launches": timed_launches,
            "clocks": sampler.summary(),
        }
        if cpu_base is not None:
            line["cpu_baseline"] = cpu_base
        if sustained is not None:
            line["sustained"] = sustained
        if gather is not None:
            line["config4_gather_check"] = gather
        line["configs"] = configs
        line["next_rows"] = extras
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, x_prev, B_global, rank):
    """Write what the last timed step returned to its caller, the sampled tokens x_{t-1} of the whole job, as
    `out_dir/x_prev.npy` (float64 [videos, tokens], token ids are exact).  The inputs, the Philox seed and the offset of the
    last step depend only on the arguments, so two builds run with the same arguments can be compared token for token.
    A job larger than 64 MB of such tokens is written as a fixed, seeded sample of whole videos, in video order."""
    import numpy as np
    import torch

    import d3pm_b200
    tokens = d3pm_b200.gather_tokens(x_prev, B_global)  # every rank takes part in the all-gather
    max_videos = (64 << 20) // (8 * tokens.shape[1])
    if tokens.shape[0] > max_videos:
        keep = torch.randperm(tokens.shape[0], generator=torch.Generator().manual_seed(0))[:max_videos].sort().values
        tokens = tokens[keep.to(tokens.device)]
    if rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        np.save(os.path.join(out_dir, "x_prev.npy"), tokens.cpu().numpy().astype(np.float64))


def _timed_steps(fn, n, dev, warm=3):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(warm):
        fn(i)
    torch.cuda.synchronize(dev)
    e0.record()
    for i in range(n):
        fn(warm + i)
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / n


def measure_config4_strong(dev, model, table, world, rank, barrier, total_videos=128, steps=40):
    """BASELINE config 4: the SAME 128 videos split over the ranks (128 / 64 / 32 / 16 per GPU at 1 / 2 / 4 / 8 GPUs), one
    fused step, device-resident, max over ranks.  (Inputs are regenerated from the global per-video seeds.)"""
    import torch
    import torch.distributed as dist
    from d3pm_b200 import _lib, ops
    import d3pm_b200

    if total_videos % world:
        return {"skipped": f"{total_videos} videos do not split over {world} ranks"}
    N, K = N_TOKENS, K_CODES
    B = total_videos // world
    b0, _ = d3pm_b200.shard_range(total_videos, world, rank)
    p_mask = float(model.log_cumprod_ct[T_NOW].exp())
    lc = torch.empty(B, N, K, device=dev)
    lu = torch.empty(B, N, K, device=dev)
    x = torch.empty(B, N, dtype=torch.int64, device=dev)
    for i in range(B):
        lc[i], lu[i], x[i] = _video_inputs(b0 + i, N, K, p_mask, dev)
    t = torch.full((B,), T_NOW, dtype=torch.int64, device=dev)
    out = torch.empty_like(x)
    barrier()
    ms = _timed_steps(lambda i: ops.fused_step(lc, lu, x, t, table, guidance_scale=GUIDANCE, sample_mode=_lib.SAMPLE_PHILOX, seed=7,
                                               offset=i, row_offset=b0 * N, x_prev_out=out), steps, dev)
    tm = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    ms = float(tm[0])
    del lc, lu
    torch.cuda.empty_cache()
    return {"what": f"config 4 (strong scaling): {total_videos} videos in total, {B} per GPU on {world} GPU(s), one fused step, "
                    f"device-resident, max over ranks", "videos_per_gpu": B, "ms_per_step": ms, "steps": steps,
            "value": total_videos * N / (ms * 1e-3), "unit": UNIT, "GBps_per_gpu": B * N * BYTES_PER_TOKEN / (ms * 1e-3) / 1e9}


def measure_config5(dev, model, table, videos=64, steps=30):
    """BASELINE config 5: MSRVTT text-conditioned shape, 64 videos x 4096 tokens, guidance on / off, one fused step."""
    import torch
    from d3pm_b200 import _lib, ops
    N, K = N_TOKENS, K_CODES
    gen = torch.Generator(device=dev).manual_seed(5)
    lc = torch.randn(videos, N, K, device=dev, generator=gen)
    lu = torch.randn(videos, N, K, device=dev, generator=gen)
    p_mask = float(model.log_cumprod_ct[T_NOW].exp())
    x = torch.where(torch.rand(videos, N, device=dev, generator=gen) < p_mask, torch.full((videos, N), K, device=dev),
                    torch.randint(0, K, (videos, N), device=dev, generator=gen))
    t = torch.full((videos,), T_NOW, dtype=torch.int64, device=dev)
    out = torch.empty_like(x)
    peak = 6554.2
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(peaks_path):
        peak = float(json.load(open(peaks_path))["hbm_gbs"])
    res = {"what": f"config 5: {videos} videos x {N} tokens x {K}+1 classes, one fused step, guidance on (scale {GUIDANCE:g}) and off "
                   f"(predict_start only), device-resident, one B200"}
    for name, u, bytes_per_token in (("guidance_on", lu, 2 * K * 4 + 16), ("guidance_off", None, K * 4 + 16)):
        time.sleep(1.0)
        ms = _timed_steps(lambda i: ops.fused_step(lc, u, x, t, table, guidance_scale=GUIDANCE, sample_mode=_lib.SAMPLE_PHILOX, seed=9,
                                                   offset=i, x_prev_out=out), steps, dev)
        gbps = videos * N * bytes_per_token / (ms * 1e-3) / 1e9
        res[name] = {"ms_per_step": ms, "value": videos * N / (ms * 1e-3), "unit": UNIT, "GBps_algorithmic": gbps,
                     "frac_of_measured_peak": gbps / peak, "bytes_per_token": bytes_per_token}
    del lc, lu
    torch.cuda.empty_cache()
    return res


def measure_k2048(dev, videos=32, steps=30):
    """The codebook the reference's UCF job configures for the denoiser (dalle num_embed 2048, SURVEY §8 a): 32 videos x 4096
    tokens x 2048 codes (the same 2.15 GB as config 2), guidance on, one fused step."""
    import torch
    import d3pm_b200
    from d3pm_b200 import _lib, ops
    N, K = N_TOKENS, 2048

    class _Stub(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.content_emb = type("E", (), {"num_embed": K + 1})()

    model = d3pm_b200.FusedDiffusionTransformer(transformer=_Stub(), diffusion_step=T_STEPS, alpha_init_type="alpha1",
                                                guidance_scale=GUIDANCE, content_seq_len=N).to(dev)
    table = model.coef_table()
    gen = torch.Generator(device=dev).manual_seed(6)
    lc = torch.randn(videos, N, K, device=dev, generator=gen)
    lu = torch.randn(videos, N, K, device=dev, generator=gen)
    p_mask = float(model.log_cumprod_ct[T_NOW].exp())
    x = torch.where(torch.rand(videos, N, device=dev, generator=gen) < p_mask, torch.full((videos, N), K, device=dev),
                    torch.randint(0, K, (videos, N), device=dev, generator=gen))
    t = torch.full((videos,), T_NOW, dtype=torch.int64, device=dev)
    out = torch.empty_like(x)
    time.sleep(1.0)
    ms = _timed_steps(lambda i: ops.fused_step(lc, lu, x, t, table, guidance_scale=GUIDANCE, sample_mode=_lib.SAMPLE_PHILOX, seed=9,
                                               offset=i, x_prev_out=out), steps, dev)
    peak = 6554.2
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(peaks_path):
        peak = float(json.load(open(peaks_path))["hbm_gbs"])
    gbps = videos * N * (2 * K * 4 + 16) / (ms * 1e-3) / 1e9
    del lc, lu
    torch.cuda.empty_cache()
    return {"what": f"{videos} videos x {N} tokens x {K}+1 classes (the UCF job's denoiser codebook), guidance {GUIDANCE:g}, one fused step, "
                    f"device-resident, one B200", "ms_per_step": ms, "value": videos * N / (ms * 1e-3), "unit": UNIT,
            "GBps_algorithmic": gbps, "frac_of_measured_peak": gbps / peak}


def measure_16bit(dev, model, table, videos=VIDEOS_PER_GPU, steps=30):
    """Config 2 with the logits a denoiser under torch.autocast produces (float16 / bfloat16): the stream kernel reads them in
    place (half the bytes), next to what such a caller paid before - `.float()` of both tensors, then the fp32 step."""
    import torch
    from d3pm_b200 import _lib, ops
    N, K = N_TOKENS, K_CODES
    gen = torch.Generator(device=dev).manual_seed(8)
    p_mask = float(model.log_cumprod_ct[T_NOW].exp())
    x = torch.where(torch.rand(videos, N, device=dev, generator=gen) < p_mask, torch.full((videos, N), K, device=dev),
                    torch.randint(0, K, (videos, N), device=dev, generator=gen))
    t = torch.full((videos,), T_NOW, dtype=torch.int64, device=dev)
    out = torch.empty_like(x)
    peak = 6554.2
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(peaks_path):
        peak = float(json.load(open(peaks_path))["hbm_gbs"])
    res = {"what": f"config 2 shape ({videos} videos x {N} tokens x {K}+1 classes, guidance {GUIDANCE:g}) with 16-bit logits: read in "
                   f"place by step_stream_kernel<4, 8, true, false, F16|BF16> (2*K*2 + 16 = {2 * K * 2 + 16} B per token update), vs. "
                   f"casting both tensors to fp32 first; tokens identical (tests/test_gpu_stream.py)"}
    for name, dt in (("float16", torch.float16), ("bfloat16", torch.bfloat16)):
        lc = torch.randn(videos, N, K, device=dev, generator=gen).to(dt)
        lu = torch.randn(videos, N, K, device=dev, generator=gen).to(dt)
        time.sleep(1.0)
        ms = _timed_steps(lambda i: ops.fused_step(lc, lu, x, t, table, guidance_scale=GUIDANCE, sample_mode=_lib.SAMPLE_PHILOX, seed=9,
                                                   offset=i, x_prev_out=out), steps, dev)
        ms_cast = _timed_steps(lambda i: ops.fused_step(lc.float(), lu.float(), x, t, table, guidance_scale=GUIDANCE,
                                                        sample_mode=_lib.SAMPLE_PHILOX, seed=9, offset=i, x_prev_out=out), 10, dev)
        gbps = videos * N * (2 * K * 2 + 16) / (ms * 1e-3) / 1e9
        res[name] = {"ms_per_step": ms, "value": videos * N / (ms * 1e-3), "unit": UNIT, "GBps_algorithmic": gbps,
                     "frac_of_measured_peak": gbps / peak, "ms_per_step_cast_then_fp32_step": ms_cast}
        if dt is torch.float16:  # the same from pinned HOST logits through the C handle (d3pm_host_step_set_logits_dtype): half of `e2e`'s bytes
            host = ops.HostStep(videos, N, K, table, guidance=True, T=T_STEPS, logits_dtype=dt)
            h_c, h_u, h_x, h_t = lc.cpu().pin_memory(), lu.cpu().pin_memory(), x.cpu().pin_memory(), t.cpu().pin_memory()
            ms_h = _timed_steps(lambda i: host(h_c, h_u, h_x, h_t, guidance_scale=GUIDANCE, seed=9, offset=i), 5, dev, warm=2)
            res["e2e_host_float16_logits"] = {"ms_per_step": ms_h, "value": videos * N / (ms_h * 1e-3), "unit": UNIT,
                                              "h2d_bytes_per_step": host.h2d_bytes, "d2h_bytes_per_step": host.d2h_bytes,
                                              "what": "d3pm_host_step_run on float16 host logits (a caller whose denoiser emits half precision): "
                                                      "informational, the headline e2e stays the fp32 workload"}
            host.close()
            del h_c, h_u
        del lc, lu
    torch.cuda.empty_cache()
    return res


def measure_decode(dev):
    """SURVEY §8 f4, the step after the path: VQVAE.decode of the sampled tokens at the shipped shape (tools/decode_bench.py) -
    the reference's PyTorch decoder on this GPU next to the native chain (tcgen05 implicit-GEMM convolutions)."""
    from tools import decode_bench
    res = decode_bench.run(videos=VIDEOS_PER_GPU, dev=dev, reps=5, quiet=True)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if "native_fp32_ms" in res and os.path.isfile(peaks_path):
        bf16 = float(json.load(open(peaks_path)).get("bf16_tflops", 0.0))
        if bf16:
            res["roofline"] = {"bound": "tensor", "unit": "TFLOP/s", "peak": 0.5 * bf16,
                               "peak_source": "half of MEASURED_PEAKS.json bf16_tflops (TF32 runs at half the bf16 rate)",
                               "achieved_fp32_mode": 3.0 * res["native_fp32_useful_TFLOPs"], "achieved_tf32_mode": res["native_tf32_useful_TFLOPs"],
                               "frac_fp32_mode": 3.0 * res["native_fp32_useful_TFLOPs"] / (0.5 * bf16),
                               "frac_tf32_mode": res["native_tf32_useful_TFLOPs"] / (0.5 * bf16),
                               "note": "fp32 mode issues three TF32 products per useful multiply-add (3xTF32), whole chain incl. attention, "
                                       "col2im and launch gaps"}
    return res


def measure_config3(dev, window=2):
    """BASELINE config 3 with the reference's REAL denoiser (tools/config3.py): the reference's own sample loop on this GPU
    against the drop-in class with the same weights, over a window of reverse steps, scaled to the 100-step chain."""
    from baseline import reference_loader as RL
    if not RL.reference_available():
        return {"skipped": "reference not staged on this box (baseline/_ref absent)"}
    from tools import config3
    return config3.run(B=VIDEOS_PER_GPU, grid=GRID, K=K_CODES, T=T_STEPS, window=window, dev=dev, guidance=GUIDANCE, quiet=True)


_NEXT_ROWS_LOGITS = None


def measure_next_rows(dev, model, table, x_t, t, x_prev, reps=20):
    """CUDA-event timings of the SURVEY §8 (f) rows at the bench shape: the denoiser head folded into the update
    (d3pm_head_step, hidden states in, tokens out) next to head-in-torch + d3pm_fused_step, and the training loss with its
    gradient (d3pm_train_rows, one pass) at the shipped training shape (16 x 1024 tokens)."""
    import torch

    from d3pm_b200 import _lib, head, ops, train

    B, N = x_t.shape
    K, D = K_CODES, 64
    gen = torch.Generator(device=dev).manual_seed(77)
    to_logits = torch.nn.Sequential(torch.nn.LayerNorm(D), torch.nn.Linear(D, K)).to(dev)
    hw = head.HeadWeights.from_module(to_logits)
    hc = torch.randn(B, N, D, device=dev, generator=gen)
    hu = torch.randn(B, N, D, device=dev, generator=gen)
    scratch = head.head_scratch(B, N, dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn, n):
        for i in range(3):
            fn(i)
        e0.record()
        for i in range(n):
            fn(3 + i)
        e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / n

    fused = timed(lambda i: head.head_step(hw, hc, hu, x_t, t, table, guidance_scale=GUIDANCE, seed=5, offset=i,
                                           x_prev_out=x_prev, scratch=scratch), reps)

    def unfused(i):
        with torch.no_grad():
            lc, lu = to_logits(hc), to_logits(hu)
        ops.fused_step(lc, lu, x_t, t, table, guidance_scale=GUIDANCE, sample_mode=_lib.SAMPLE_PHILOX, seed=5, offset=i,
                       x_prev_out=x_prev)

    unf = timed(unfused, 5)
    Bt, Nt = 16, 1024
    logits = torch.randn(Bt, Nt, K, device=dev, generator=gen)
    x0 = torch.randint(0, K, (Bt, Nt), device=dev, generator=gen)
    tt = torch.randint(0, T_STEPS, (Bt,), device=dev, generator=gen)
    xt = model.q_sample_tokens(x0, tt)
    w = torch.ones(Bt, device=dev)
    tr = timed(lambda i: train._train_rows(logits, K, x0, xt, tt, table, (1, 1), backward=2, w_main=w, w_aux=w, want_recon=True), reps)
    qs = timed(lambda i: train.q_sample_tokens(x0, tt, model._sched8(), K, seed=3, offset=i), reps)
    # purity-prior step (prior_rule 2): candidate draw + purity on the bench's own logits, then the per-video reveal
    lc, lu = _NEXT_ROWS_LOGITS
    pur = {}

    def purity(i):
        pur["o"] = ops.fused_step(lc, lu, x_t, t, table, guidance_scale=GUIDANCE, sample_mode=_lib.SAMPLE_PHILOX, seed=5, offset=i,
                                  sample_from=_lib.FROM_RECON, want_score=True)

    pd = timed(purity, reps)
    n_reveal = torch.full((B,), 40, dtype=torch.int32, device=dev)
    ps = timed(lambda i: ops.purity_select(x_t, pur["o"]["x_prev"], pur["o"]["score"], n_reveal, K, seed=1, offset=i), reps)
    # the host entry of the fused head: pinned host HIDDEN STATES in, host tokens out (d3pm_host_head_step_run) - the boundary
    # a deployment whose denoiser runs elsewhere would use: 64x fewer bytes on the bus than the logits
    hh = ops.HostStep(B, N, K, table, guidance=True, T=T_STEPS, hidden_dim=D)
    h_hc, h_hu = hc.cpu().pin_memory(), hu.cpu().pin_memory()
    h_x, h_t = x_t.cpu().pin_memory(), t.cpu().pin_memory()
    e2e_head = timed(lambda i: hh.head(hw, h_hc, h_hu, h_x, h_t, guidance_scale=GUIDANCE, seed=5, offset=i), 10)
    head_h2d, head_d2h = hh.h2d_bytes, hh.d2h_bytes
    hh.close()
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    bf16_peak = float(json.load(open(peaks_path)).get("bf16_tflops", 0.0)) if os.path.isfile(peaks_path) else 0.0
    mma_flops = 2.0 * B * N * K * D * (1 + 3)  # statistics pass in 1xTF32, sampling pass in 3xTF32
    return {
        "e2e_host_hidden_states": {"ms_per_step": e2e_head, "value": B * N / (e2e_head * 1e-3), "unit": UNIT,
                                   "h2d_bytes_per_step": head_h2d, "d2h_bytes_per_step": head_d2h,
                                   "what": "C ABI d3pm_host_head_step_run: pinned host hidden states [B, N, 64] x2 -> fused head + "
                                           "update -> host tokens, copies inside the timed region"},
        "purity_prior_step": {"ms_candidate_draw_and_purity": pd, "ms_reveal": ps,
                              "what": "p_sample with prior_rule 2: d3pm_fused_step (D3PM_FROM_RECON + score, stream kernel) + d3pm_purity_select"},
        "q_sample_tokens": {"ms_per_step": qs, "what": "d3pm_q_sample_tokens, 16 x 1024 tokens: forward noising of the training step, one kernel"},
        "head_fused_step": {"ms_per_step": fused, "token_updates_per_s": B * N / (fused * 1e-3), "valid_weight_bound": bool(hw.valid),
                            "tf32_TFLOPs_issued": mma_flops / (fused * 1e-3) / 1e12, "useful_fp32_TFLOPs": 2.0 * B * N * K * D * 2 / (fused * 1e-3) / 1e12,
                            "measured_bf16_peak_TFLOPs": bf16_peak,
                            "tf32_frac_of_half_bf16_peak": (mma_flops / (fused * 1e-3) / 1e12) / (0.5 * bf16_peak) if bf16_peak else None,
                            "what": "d3pm_head_step: LayerNorm + Linear(64 -> 4096) of both denoiser passes + the whole update, "
                                    "tcgen05 (statistics pass 1xTF32, sampling pass 3xTF32), logits never in memory"},
        "head_in_torch_then_fused_step": {"ms_per_step": unf, "what": "torch LayerNorm + Linear (fp32) x2, then d3pm_fused_step"},
        "train_loss_and_gradient": {"ms_per_step": tr, "GBps_algorithmic": 2 * Bt * Nt * K * 4 / tr / 1e6,
                                    "what": "d3pm_train_rows backward=2, 16 x 1024 tokens x 4096 codes, losses + logits gradient in one pass"},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300,
                    help="timed steps of the headline metric (`value`, `ms_per_step`); the default (0.1 s) is a burst "
                         "measurement.  The other blocks keep their own counts, reported beside them: `e2e` times "
                         "min(steps, 10) steps (at least 3), `sustained` a fixed 1500 (power-capped on B200)")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--global-videos", type=int, default=0,
                    help="strong scaling: this many videos in total, split over the ranks (config 4: 128); "
                         "default 0 = weak scaling, 16 videos per GPU")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the tokens the last timed step sampled to DIR/x_prev.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the tokens of --impl ours")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
