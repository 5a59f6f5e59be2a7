#!/usr/bin/env python
"""SAC learner hot-path benchmark (BASELINE.json metric: SAC updates/sec, Humanoid-v5 shape, B=256; PER samples/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (N=1) = BASELINE.json configs[1]: Humanoid-v5 SAC update (obs 348, act 17, 3x512 networks_model2 MLPs,
batch 256) over a 1M-transition prioritized replay ring resident in HBM.  One STEP = what the trainer loop does
per environment step on the learner side: prioritized sample of 256 (index draw + IS weights + gather) -> one
full update_parameters (target, twin-critic, actor, temperature, Adam, Polyak) -> priority write-back.

  value : steps/s with every input resident in HBM (uniforms / eps drawn on device), CUDA events on the
          library's stream, no host sync inside the timed region.
  e2e   : steps/s through the public API (`replay_buffer.push` of one fresh transition + `update_parameters(256)`
          with host-drawn uniforms copied H2D and the three losses read back D2H every step).
  N>1   : independent replicas (one agent per GPU, no collective: the single-agent path does not shard), weak scaling.
  sharded : the two modes north_star shards (SURVEY 8e), measured in the same run at the same N and reported in the line's
          `sharded` object: C5 population (128 agents per GPU = 1024 on 8, batched fused updates, no inter-GPU traffic) and
          C4 large-batch data parallel (global batch 8192 and 65536 split over the N ranks, gradient all-reduce over NVLink).
  --impl reference : the CPU restatement of the reference (numpy/OpenBLAS update + C PER sampler) on the host cores.
  --dump-outputs DIR : after the K timed steps of `value`, the arrays their last step computed (losses, alpha, network
          parameters, priority table) as DIR/<name>.npy; the seeded inputs make two builds comparable output for output.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

OBS, ACT, HID, NH, B = 348, 17, 512, 3, 256
CAPACITY = 1_000_000
FLOP_PER_UPDATE = 5.382e9          # SURVEY 8d: fwd + necessary bwd, B=256, C2 shapes
WORKLOAD = "Humanoid-v5 SAC update obs348/act17/hidden512x3 (networks_model2) B=256 + 1M-transition prioritized replay"


def synth_transitions(n, seed):
    rng = np.random.RandomState(seed)
    s = rng.standard_normal((n, OBS)).astype(np.float32)
    a = rng.uniform(-0.4, 0.4, (n, ACT)).astype(np.float32)
    r = rng.standard_normal(n).astype(np.float32)
    s2 = rng.standard_normal((n, OBS)).astype(np.float32)
    d = (rng.uniform(size=n) < 0.01).astype(np.float32)
    return s, a, r, s2, d


def synth_priorities(n, seed):
    return (np.abs(np.random.RandomState(seed).standard_normal(n)) + 1e-6).astype(np.float32)


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe): NVML polled every ~4 ms from a
    thread (the timed region of a default run is ~70 ms, too short for `nvidia-smi -lms`), `nvidia-smi` as the fallback."""

    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))

    def __init__(self, gpu):
        self.gpu, self.sm, self.mx, self.reasons, self.proc, self.stop, self.thread, self.rows = gpu, [], [], set(), None, False, None, []
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[gpu]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else gpu
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.mx.append(float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)))
        except Exception:
            self.nvml = None

    def sample_now(self):
        """One sample from the calling thread (the bench calls it while the queued steps are still running on the GPU)."""
        n = self.nvml
        if not n:
            return
        try:
            self.sm.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
            mask = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
            for bit, name in self.REASONS:
                if mask & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def _poll(self):
        while not self.stop:
            self.sample_now()
            time.sleep(0.004)

    def __enter__(self):
        if self.nvml:
            self.sample_now()                       # absorbs NVML's slow first queries before the timed region starts ...
            self.sm.clear(); self.reasons.clear()   # ... and is not a sample of it
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return self
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            r = [x.strip() for x in line.split(",")]
            if len(r) >= 7 and r[0].replace(".", "").isdigit():
                self.sm.append(float(r[0])); self.mx.append(float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        self.reasons.add(name)

    def __exit__(self, *a):
        self.stop = True
        if self.thread:
            self.thread.join(timeout=1.0)
        if self.proc:
            self.proc.terminate()

    def summary(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                "reasons": sorted(self.reasons), "samples": len(self.sm), "source": "nvml" if self.nvml else "nvidia-smi"}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return p, "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


# ------------------------------------------------------------------------------------------------------------------
# reference arm: CPU restatement of the reference on the host cores (the oracle; bench is allowed to time it)
# ------------------------------------------------------------------------------------------------------------------
_CPU_DATA = {}


def cpu_reference(steps, warmup, n_per=CAPACITY, seed=0, threads=None):
    """The workload of our arm on the host: PER sample at N = 1M (replay_buffer.py:48-68) -> gather of 256 rows out of a 1M-row
    host ring -> IS-weighted update (sac_imp.py:74-144 + the per_weighted_loss extension our arm runs) -> priority write-back."""
    from oracle import per_oracle as PO
    from oracle import sac_oracle_np as O
    threads = os.cpu_count() if threads is None else threads
    limiter = None
    try:    # torchrun exports OMP_NUM_THREADS=1, which would handicap the CPU arm: set the BLAS pool explicitly
        from threadpoolctl import threadpool_limits
        limiter = threadpool_limits(limits=threads)
    except Exception:
        pass
    st = O.make_state(OBS, ACT, HID, NH, seed=seed, head_scale=0.25)
    pri = synth_priorities(n_per, seed)
    pa = PO.pow_alpha(pri)
    if "ring" not in _CPU_DATA:      # 1M-row gather source like ours (the same 125k-row block eight times): 2.9 GB of host memory
        chunk = 125_000
        s, a, r, s2, d = synth_transitions(chunk, seed)
        reps = CAPACITY // chunk
        _CPU_DATA["ring"] = tuple(np.tile(x, (reps, 1)) if x.ndim == 2 else np.tile(x, reps) for x in (s, a, r, s2, d))
    s, a, r, s2, d = _CPU_DATA["ring"]
    rng = np.random.RandomState(seed + 1)

    def step(i):
        u = rng.random_sample(B)
        idx, w = PO.sample(pa, u, PO.beta(1 + i))                                  # replay_buffer.py:48-68 at N = 1M
        batch = dict(s=s[idx], a=a[idx], r=r[idx], s2=s2[idx], d=d[idx],
                     eps_next=rng.standard_normal((B, ACT)).astype(np.float32), eps_cur=rng.standard_normal((B, ACT)).astype(np.float32))
        _, aux = O.update_parameters(st, batch, per_weights=w, return_aux=True)     # sac_imp.py:74-144
        td = np.abs(aux["td1"]).astype(np.float32)
        PO.update_priorities(pri, idx, td)                                          # replay_buffer.py:84-87
        pa[idx] = PO.pow_alpha(pri[idx])

    for i in range(warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(steps):
        step(warmup + i)
    dt = time.perf_counter() - t0
    try:
        from threadpoolctl import threadpool_info
        cores = max([p.get("num_threads", 1) for p in threadpool_info()] + [1])
    except Exception:
        cores = threads
    if limiter is not None:
        limiter.restore_original_limits()
    return steps / dt, dt / steps * 1e3, cores


def cpu_thread_sweep(steps, warmup):
    """SURVEY 8d: threads in {1, all host cores}; the best is the baseline, both are reported."""
    runs = []
    for t in sorted({1, os.cpu_count() or 1}):
        ups, ms, cores = cpu_reference(steps, warmup, threads=t)
        runs.append({"threads": t, "updates_per_s": ups, "ms_per_step": ms, "blas_threads_seen": cores})
    best = max(runs, key=lambda r: r["updates_per_s"])
    return best, runs


def bench_config(args, world):
    """`config` of the JSON line: shared by both arms (the driver compares them)."""
    return {"workload": WORKLOAD, "launch": args.launch, "math": args.math, "replicas": world,
            "step": "sample(256) -> update -> priority write-back, " + ("sequential on one stream" if args.no_pipeline else
                    "software-pipelined: write-back and the next sample run on a second stream under the tail of the update (sacb_per_step; bitwise equal to the sequential order)"),
            "l2_policy": "inputs larger than L2: 1M-row ring (2.9 GB) + 4 MB priority table re-read every step; weights/Adam state (63 MB) stay L2 resident by design"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = args.steps
    warmup = max(3, min(args.warmup, 50))
    best, runs = cpu_thread_sweep(steps, warmup)
    ups, ms = best["updates_per_s"], best["ms_per_step"]
    sample = f"{steps} steps of the full workload (PER sample at N=1M + 1M-row gather + IS-weighted update + priority write-back), {warmup} warm-up, threads in {{1, all}}: best"
    line = {"impl": "reference", "metric": "SAC updates/sec (Humanoid-v5 shape, B=256, 1M-transition PER)", "value": ups, "unit": "updates/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": bench_config(args, int(os.environ.get("WORLD_SIZE", "1"))),
            "cpu_baseline": {"value": ups, "unit": "updates/s", "cores": best["threads"], "host_cores": os.cpu_count(), "kind": "port", "sample": sample, "thread_sweep": runs},
            "e2e": {"value": ups, "unit": "updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------------------
def build_agent(hw, device, launch, math, seed):
    import torch
    hw.use_networks("model2")
    torch.manual_seed(seed)
    agent = hw.SAC(OBS, ACT, hidden_dim=HID, device=f"cuda:{device}", replay="per", capacity=CAPACITY, max_batch=B,
                   math=math, launch=launch, seed=seed, per_weighted_loss=True)
    # shrink the policy heads like the parity cases do: keeps tanh out of saturation on N(0,1) observations
    with torch.no_grad():
        agent.policy.mean.weight.mul_(0.25)
        agent.policy.log_std.weight.mul_(0.25)
    chunk = 125_000
    s, a, r, s2, d = synth_transitions(chunk, seed)
    for _ in range(CAPACITY // chunk):
        agent.replay_buffer.push_many(s, a, r, s2, d)
    agent.replay_buffer.set_priorities(synth_priorities(CAPACITY, seed))
    return agent


def dump_outputs(N, agent, out_dir):
    """What the timed steps computed, as float32 .npy files, so that two builds can be compared output for output: the three
    losses of the last update, alpha and log_alpha, every parameter of the five networks (3.6 M floats) and the 1M-entry priority
    table the last write-back updated; 18 MB in all.  Every input is seeded: the same arguments give the same inputs in every run."""
    os.makedirs(out_dir, exist_ok=True)
    losses = np.zeros(3, np.float32)
    N.check(N.lib().sacb_get_losses(agent._h, 0, N.ptr(losses)))
    sc = agent._scalars()
    out = {"losses": losses, "alpha": np.array([sc.alpha], np.float32), "log_alpha": np.array([sc.log_alpha], np.float32),
           "priorities": agent.replay_buffer.priorities}
    with agent._library_stream():
        for net in ("policy", "q1", "q2", "q1_target", "q2_target"):
            for k, v in getattr(agent, net).state_dict().items():
                out[f"{net}.{k}"] = v.detach().cpu().numpy().astype(np.float32)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def eager_cuda_baseline(device, steps=100):
    """SURVEY 8d's like-for-like GPU bar: the reference's update as stock PyTorch eager on this B200 (oracle/sac_ref_torch.py, a
    plain autograd restatement pinned to the same golden vectors), and the full learner step as the reference would run it with
    device='cuda': prioritized sampling in host numpy at N = 1M (replay_buffer.py:48-87 keeps the buffer on the host) + H2D + update."""
    import torch
    from oracle import sac_oracle_np as O
    from oracle import sac_ref_torch as T
    st = O.make_state(OBS, ACT, HID, NH, seed=0, head_scale=0.25)
    agent = T.TorchSAC(st, f"cuda:{device}")
    rng = np.random.RandomState(3)
    s, a, r, s2, d = synth_transitions(8192, 3)
    dev = agent.device
    ts, ta, ts2 = (torch.as_tensor(x, device=dev) for x in (s, a, s2))
    tr, td_ = torch.as_tensor(r, device=dev).reshape(-1, 1), torch.as_tensor(d, device=dev).reshape(-1, 1)

    def upd(i):
        j = torch.randint(0, 8192, (B,), device=dev)
        return agent.update(ts[j], ta[j], tr[j], ts2[j], td_[j])      # eps via torch.randn_like, 3 .item() syncs (sac_imp.py:141-143)

    for i in range(10):
        upd(i)
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for i in range(steps):
        upd(i)
    torch.cuda.synchronize(dev)
    upd_ms = (time.perf_counter() - t0) / steps * 1e3
    per = T.NumpyPER(synth_priorities(CAPACITY, 0))
    hs, ha, hr, hs2, hd = _CPU_DATA.get("ring") or tuple(np.tile(x, (CAPACITY // 8192 + 1, 1))[:CAPACITY] if x.ndim == 2 else np.tile(x, CAPACITY // 8192 + 1)[:CAPACITY] for x in (s, a, r, s2, d))
    n_full = max(5, min(20, steps // 5))

    def full(i):
        idx, w = per.sample(B)                                         # host numpy, O(N) per call
        f = lambda x, col=False: torch.FloatTensor(x[idx]).to(dev).reshape(-1, 1) if col else torch.FloatTensor(x[idx]).to(dev)      # sac_imp.py:81-85
        _, tdv = agent.update(f(hs), f(ha), f(hr, True), f(hs2), f(hd, True), weights=torch.as_tensor(w, device=dev).reshape(-1, 1))
        per.update_priorities(idx, tdv.reshape(-1).cpu())

    full(0)
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for i in range(n_full):
        full(i)
    torch.cuda.synchronize(dev)
    full_ms = (time.perf_counter() - t0) / n_full * 1e3
    return {"kind": "port (plain torch autograd restatement of sac_imp.py:74-144, stock PyTorch eager kernels, device=cuda on this B200)",
            "update_only": {"value": 1e3 / upd_ms, "unit": "updates/s", "ms_per_update": upd_ms, "steps": steps},
            "full_step": {"value": 1e3 / full_ms, "unit": "updates/s", "ms_per_step": full_ms, "steps": n_full,
                          "what": "numpy PER sample at N=1M on the host (as the reference keeps its buffer) + H2D of the minibatch + eager update + priority write-back"},
            "torch": torch.__version__}


def bench_population(hw, local, world, rank, dist, red_dev, agents_per_gpu=128, steps=10):
    """C5 (BASELINE.json configs[4]): 1024 independent Humanoid agents over 8 B200 = 128 agents per GPU, weak scaling; every agent
    owns a uniform replay ring of 100k transitions in HBM (1024 x 100k x 2860 B = 293 GB over 8 GPUs = 36.6 GB per GPU; 16k of
    them resident at bench time, far beyond L2 in total), positions and eps drawn on the device, no inter-GPU traffic."""
    import gc
    import torch
    N = hw._native
    lib = N.lib()
    first = rank * agents_per_gpu
    cap, fill = 100_000, 16_384
    hw.use_networks("model2")
    pop = hw.PopulationSAC(agents_per_gpu, OBS, ACT, hidden_dim=HID, device=f"cuda:{local}", seeds=list(range(first, first + agents_per_gpu)),
                           capacity=cap, max_batch=B, seed=1000 + rank)
    s, a, r, s2, d = synth_transitions(fill, 100 + rank)
    for i in range(agents_per_gpu):
        pop.push_many(i, s, a, r, s2, d)
    for _ in range(3):
        pop.update_parameters(B, sync=False)
    pop.synchronize()
    if world > 1:
        dist.barrier()
    ms = ctypes.c_float()
    N.check(lib.sacb_timer_start(pop._h))
    for _ in range(steps):
        pop.update_parameters(B, sync=False)
    N.check(lib.sacb_timer_stop(pop._h, ctypes.byref(ms)))
    losses = pop.update_parameters(B)
    t = torch.tensor([ms.value], device=red_dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    per_step = float(t.item()) / steps
    ups = world * agents_per_gpu / (per_step * 1e-3)
    peaks, _ = measured_peaks()
    out = {"config": "BASELINE.json configs[4]: population of independent Humanoid-v5 (obs348/act17/512x3) SAC agents, B=256, one batched fused update program per step",
           "agents_per_gpu": agents_per_gpu, "agents_total": agents_per_gpu * world, "ms_per_population_step": per_step,
           "agent_updates_per_s": ups, "agent_updates_per_s_per_gpu": ups / world, "scaling": "weak", "collective": "none",
           "ring": f"per-agent uniform ring, capacity {cap} transitions in HBM ({cap * agents_per_gpu * 2860 / 1e9:.1f} GB per GPU), {fill} resident per agent at bench time; positions drawn on the device",
           "algorithmic_TFLOPs_per_gpu": ups / world * FLOP_PER_UPDATE / 1e12,
           "roofline": {"bound": "hbm", "achieved": ups / world * 63.7e6 / 1e9, "peak": float(peaks.get("hbm_gbs", 6650.0)), "unit": "GB/s",
                        "frac": ups / world * 63.7e6 / 1e9 / float(peaks.get("hbm_gbs", 6650.0)),
                        "note": "algorithmic bytes = 63.0 MB of learner state streamed once + 0.73 MB gather per agent-update (SURVEY 8d: 85 FLOP/B, HBM-bound)"},
           "finite_losses": bool(np.isfinite([v for l in losses for v in l.values()]).all())}
    del pop
    gc.collect()
    return out


def bench_data_parallel(hw, local, world, rank, dist, red_dev, global_batch, steps):
    """C4 (BASELINE.json configs[3]): one replicated agent, global batch split over the ranks, two dependent gradient all-reduces per
    step (critics, then actor + temperature: sac_imp.py:107-118).  The all-reduce share is measured by timing the same steps with
    the exchange skipped (world > 1)."""
    import gc
    import torch
    N = hw._native
    lib = N.lib()
    bl, cap = global_batch // world, 65536
    hw.use_networks("model2")
    torch.manual_seed(0)                      # identical replicas
    agent = hw.SAC(OBS, ACT, hidden_dim=HID, device=f"cuda:{local}", capacity=cap, max_batch=bl, math="bf16x3", seed=100 + rank)
    with torch.no_grad():
        agent.policy.mean.weight.mul_(0.25); agent.policy.log_std.weight.mul_(0.25)
    torch.cuda.synchronize()
    s, a, r, s2, d = synth_transitions(cap, 200 + rank)
    agent.replay_buffer.push_many(s, a, r, s2, d)
    dp = hw.distributed.DataParallelSAC(agent)
    idx = np.random.RandomState(rank).randint(0, cap, bl).astype(np.int64)
    dp.update_parameters(bl, idx=idx)

    def timed(n, exchange=True):
        dp.exchange = exchange
        for _ in range(2):
            dp.update_parameters(bl, staged=True, sync=False)
        agent.synchronize()
        if world > 1:
            dist.barrier()
        ms = ctypes.c_float()
        N.check(lib.sacb_timer_start(agent._h))
        for _ in range(n):
            dp.update_parameters(bl, staged=True, sync=False)
        N.check(lib.sacb_timer_stop(agent._h, ctypes.byref(ms)))
        t = torch.tensor([ms.value], device=red_dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / n

    per = timed(steps)
    no_x = timed(steps, exchange=False) if world > 1 else per
    dp.exchange = True
    last = dp.update_parameters(bl, staged=True)
    flop = FLOP_PER_UPDATE * global_batch / 256
    peaks, _ = measured_peaks()
    peak_tf = float(peaks.get("bf16_tflops_sustained", 1400.0))
    out = {"global_batch": global_batch, "local_batch": bl, "ms_per_update": per, "updates_per_s": 1e3 / per, "transitions_per_s": global_batch / per * 1e3,
           "algorithmic_TFLOPs_total": flop / (per * 1e-3) / 1e12, "algorithmic_TFLOPs_per_gpu": flop / world / (per * 1e-3) / 1e12,
           "roofline_frac_per_gpu": flop / world / (per * 1e-3) / 1e12 / peak_tf, "exchange": dp.exchange_kind,
           "ms_without_exchange": no_x, "exchange_share": max(0.0, 1.0 - no_x / per), "finite_losses": bool(np.isfinite(list(last.values())).all())}
    del dp, agent
    gc.collect()
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist
    import humanoid_walking_with_sac_b200 as hw
    N = hw._native
    lib = N.lib()

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    backend = os.environ.get("SACB_BENCH_BACKEND", "nccl")      # "gloo": diagnosis only (timing barrier without NCCL)
    red_dev = f"cuda:{local}" if backend == "nccl" else "cpu"
    if world > 1:
        if backend == "nccl":
            dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
        else:
            dist.init_process_group(backend)
    agent = build_agent(hw, local, args.launch, args.math, seed=rank)
    torch.cuda.synchronize()
    agent._publish_alias_writes()      # build_agent scaled the heads through the torch aliases
    h = agent._h

    def device_step():
        if args.no_pipeline:      # the three calls back to back on one stream
            N.check(lib.sacb_per_sample(h, 0, None, B, None, None, None, None, None, None, None))
            N.check(lib.sacb_update(h, B, None, None, None, None, N.USE_LAST_SAMPLE | N.NO_LOSS_READBACK))
            N.check(lib.sacb_per_update_from_td(h, 0, B))
        else:                     # same work, the write-back and the next sample run under the tail of the update (second stream)
            N.check(lib.sacb_per_step(h, B, None, N.NO_LOSS_READBACK))

    def barrier():
        agent.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(3, args.warmup)):
        device_step()
    barrier()
    st0 = agent.stats()["kernel_launches"]
    ms = ctypes.c_float()
    with ClockSampler(local) as clk:
        N.check(lib.sacb_timer_start(h))
        for _ in range(args.steps):
            device_step()
        # (NVML is only queried from the sampler's own thread: a query from THIS thread between the last launch and the stop event
        #  stalled the submission of the queued steps by 30-100 ms in one run out of four)
        N.check(lib.sacb_timer_stop(h, ctypes.byref(ms)))
        if clk.nvml and not clk.sm:
            clk.sample_now()      # region shorter than one NVML query: one sample right behind it
        if not clk.nvml:
            time.sleep(0.15)
    barrier()
    launches = agent.stats()["kernel_launches"] - st0
    if args.dump_outputs and rank == 0:
        dump_outputs(N, agent, args.dump_outputs)
    if world > 1:
        print(f"[rank {rank}] device {local}: {ms.value / args.steps:.4f} ms/step", file=sys.stderr)
    t = torch.tensor([ms.value], device=red_dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    value = world * args.steps / (ms_total * 1e-3)

    # ---- roofline of the dominant kernel (the update program) measured live: update-only replays on the same stream
    upd_ms = ctypes.c_float()
    N.check(lib.sacb_time_update(h, B, max(50, args.steps), ctypes.byref(upd_ms)))
    stage_us = (ctypes.c_float * 64)()
    n_st = lib.sacb_time_stages(h, B, stage_us, 64)
    per_ms = ctypes.c_float()
    N.check(lib.sacb_timer_start(h))
    for _ in range(args.steps):
        N.check(lib.sacb_per_sample(h, 0, None, B, None, None, None, None, None, None, None))
    N.check(lib.sacb_timer_stop(h, ctypes.byref(per_ms)))
    tp = torch.tensor([per_ms.value], device=red_dev)
    if world > 1:
        dist.all_reduce(tp, op=dist.ReduceOp.MAX)
    per_call_ms = float(tp.item()) / args.steps      # max over ranks; every rank samples from its own 1 M-row table
    peaks, peak_src = measured_peaks()
    achieved_tf = FLOP_PER_UPDATE / (upd_ms.value * 1e-3) / 1e12
    peak_tf = float(peaks.get("bf16_tflops_sustained", 1400.0))
    traffic, traffic_file = None, None      # DRAM bytes of one update program (its stage kernels, warm caches) from the committed ncu capture
    for name in ("r02_update_traffic.json", "r01_update_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                traffic, traffic_file = float(json.load(f)["update_dram_bytes"]), name.replace("traffic.json", "stages_ncu.csv")
            break
        except Exception:
            pass
    roofline = {"bound": "tensor", "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf, "traffic": traffic,
                "traffic_source": "NOT measured in this run: constant read from the committed ncu capture profiles/%s: dram__bytes_read.sum + dram__bytes_write.sum summed over the stage kernels of one update (algorithmic bytes if streamed from HBM: 63.7e6; the state stays L2 resident)" % traffic_file,
                "kernel": "sac_update_kernel (one fused update program: %d launches/step in '%s' mode)" % (1 if args.launch == "persistent" else n_st, args.launch),
                "ms_per_launch_sum": upd_ms.value, "peak_source": peak_src + " bf16 dense, sustained (each product costs 3 bf16 MMAs: algorithmic FLOPs are counted once)",
                "note": "single-agent B=256 is latency/occupancy bound (SURVEY 8d): 25 dependent stages of <=0.27 GFLOP, ~3 us of fixed cost each (profiles/r02_summary.md, 'Single agent')",
                "stage_us": [round(float(stage_us[i]), 2) for i in range(max(0, min(n_st, 64)))],
                "per_sample": {"ms_per_call": per_call_ms, "samples_per_s": B / (per_call_ms * 1e-3),
                               "achieved_GBps": (3 * 4.0 * CAPACITY + B * 4 * (2 * OBS + ACT + 2)) / (per_call_ms * 1e-3) / 1e9,
                               "peak_GBps": float(peaks.get("hbm_gbs", 6650.0)), "algorithmic_bytes": "3 passes over p_alpha (4 B x N) + B rows"}}

    # ---- e2e through the public API: push one transition, update_parameters(256) with host uniforms, losses read back
    s1, a1, r1, s21, d1 = synth_transitions(args.steps + 8, 12345 + rank)
    row_bytes = int(lib.sacb_row_floats(h)) * 4
    for i in range(3):
        agent.replay_buffer.push(s1[i], a1[i], r1[i], s21[i], bool(d1[i]))
        agent.update_parameters(B)
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        agent.replay_buffer.push(s1[i], a1[i], float(r1[i]), s21[i], bool(d1[i]))
        out = agent.update_parameters(B)
    agent.synchronize()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], device=red_dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e = world * args.steps / float(te.item())

    # ---- e2e, K = 8 learner steps per call (SURVEY 8f rank 3): 8 transitions pushed through the pinned staging ring, learner_steps(k=8)
    #      (device-drawn uniforms / eps), ONE read-back of the 8 loss triples
    K = 8
    calls = max(1, args.steps // K)
    sk, ak, rk, s2k, dk = synth_transitions(K * (calls + 2), 54321 + rank)
    def k_call(c):
        for i in range(c * K, (c + 1) * K):
            agent.replay_buffer.push(sk[i], ak[i], float(rk[i]), s2k[i], bool(dk[i]))
        return agent.learner_steps(B, k=K)
    k_call(calls); k_call(calls + 1)
    barrier()
    t0 = time.perf_counter()
    for c in range(calls):
        out_k = k_call(c)
    agent.synchronize()
    tk = torch.tensor([time.perf_counter() - t0], device=red_dev)
    if world > 1:
        dist.all_reduce(tk, op=dist.ReduceOp.MAX)
    e2e_k = world * calls * K / float(tk.item())

    cpu = eager = None
    if rank == 0 and world == 1 and not args.no_cpu:
        best, runs = cpu_thread_sweep(steps=30, warmup=3)
        cpu = {"value": best["updates_per_s"], "unit": "updates/s", "cores": best["threads"], "host_cores": os.cpu_count(), "kind": "port", "thread_sweep": runs,
               "sample": "30 steps of the full workload on the host at threads in {1, all}, best reported (numpy/OpenBLAS restatement of sac_imp.py:74-144, IS-weighted like ours, + C restatement of replay_buffer.py:48-87 at N=1M, 1M-row host ring)"}
        try:
            eager = eager_cuda_baseline(local)
        except Exception as e:      # a baseline must not take the bench down
            eager = {"error": repr(e)}

    # ---- the two sharded modes at this N (SURVEY 8e); the single agent above is freed first
    sharded = None
    if not args.no_sharded:
        del agent
        import gc
        gc.collect()
        sharded = {}
        try:
            sharded["population"] = bench_population(hw, local, world, rank, dist, red_dev, agents_per_gpu=args.agents_per_gpu)
            sharded["data_parallel"] = [bench_data_parallel(hw, local, world, rank, dist, red_dev, 8192, 20),
                                        bench_data_parallel(hw, local, world, rank, dist, red_dev, 65536, 6)]
        except Exception as e:
            sharded["error"] = repr(e)

    if rank == 0:
        line = {"metric": "SAC updates/sec (Humanoid-v5 shape, B=256, 1M-transition PER)", "value": value, "unit": "updates/s", "n_gpus": world,
                "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_total / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": {"bf16x3": "f32 (bf16 hi/lo operand pairs, 3 tcgen05 MMAs per product, f32 accumulate in TMEM; f32 master weights / Adam)", "fp32": "f32 (FFMA on the bf16-pair operands)"}[args.math],
                "data": "synthetic",
                "config": bench_config(args, world),
                "e2e": {"value": e2e, "unit": "updates/s", "h2d_bytes_per_step": row_bytes + 8 * B, "d2h_bytes_per_step": 12,
                        "what": "the trainer's own call sequence (trainer.py:190-205): replay_buffer.push(one transition) + update_parameters(256) with host-drawn uniforms, three losses read back, every step; the pushed row and the uniforms cross host->device out of pinned staging blocks (read there by the push / search kernels), the losses device->host into a pinned block (stored by the last stage), inside the timed region",
                        "batched_k8": {"value": e2e_k, "unit": "updates/s", "h2d_bytes_per_step": row_bytes, "d2h_bytes_per_step": 12,
                                       "what": "8 pushes + learner_steps(256, k=8): uniforms / eps drawn on the device, one read-back of the 8 loss triples per call"}},
                "gpu_launches": int(launches), "clocks": clk.summary(), "roofline": roofline, "cpu_baseline": cpu, "eager_cuda_baseline": eager, "sharded": sharded,
                "per_samples_per_s": world * B / (per_call_ms * 1e-3),      # whole job: `world` independent prioritized buffers
                "last_losses": out}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--launch", default=os.environ.get("SACB_LAUNCH", "staged"), choices=["staged", "persistent"])
    ap.add_argument("--math", default=os.environ.get("SACB_MATH", "bf16x3"), choices=["bf16x3", "fp32"])
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-sharded", action="store_true", help="skip the population / data-parallel block")
    ap.add_argument("--agents-per-gpu", type=int, default=128)
    ap.add_argument("--no-pipeline", action="store_true", help="value: run sample / update / write-back sequentially on one stream")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
