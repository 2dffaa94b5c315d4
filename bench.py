#!/usr/bin/env python
"""bench.py -- LR event-frames/sec of the ESR hot path on B200 (BASELINE.json metric), one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg2|cfg3|cfg4] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" = one batch of B sequences x L LR event frames taken from raw events to redistributed SR events:
  encode L frames (LR->HR lift + count scatter) -> L-2 DeepRecurrNet forwards with carried ConvGRU state
  -> cnt2event of the L-2 SR count tensors.          (SURVEY.md 8d; infer_ours_cnt.py:54-75)
value   : events already resident in HBM when a timed step starts.
e2e     : the same step through the public API with pinned HOST buffers: H2D of the events and D2H of the
          resulting event lists inside the timed region.
parity  : one un-timed check per workload of the network output of the measured plan against the CPU oracle
          (all windows, carried state) -- `parity.rel_max` must stay below 1e-3 (north_star).
roofline: FLOP-weighted achieved TFLOP/s of the dominant kernel FAMILY (every tcgen05 conv launch of one step, timed
          live with CUDA events), against the measured sustained bf16 peak; `roofline_hbm` = the HBM-bound kernels
          (count scatter, redistribution, small-channel full-resolution convs) against the measured copy bandwidth.
configs : the other BASELINE.json network configurations (cfg3 4x SR; cfg4 4x SR long sequence) with their own
          value / e2e / parity / cpu_baseline; `sweep` = configs[4] (scatter + redistribute at 1e5..1e7 events).
Multi-GPU: the path shards by batch with no data-path collective (inference); every rank runs the per-GPU batch of
the workload on its own shard (weak scaling) and the time is the max over ranks.  Training (`train`) adds the one
exchange of the path: the NCCL all-reduce of the flat gradient, captured with the iteration in one CUDA graph.
`--impl reference` times the CPU restatement of the same path on the host cores (rank 0 only): the oracle port of the
network plus the reference's OWN compiled Cython redistribution (oracle/_ref) when it was built.
`--dump-outputs DIR` writes what the last timed step of the headline workload returned (rank 0): sr_counts.npy and
events.npy, float32, at most 64 MB together (a fixed seeded sample beyond that).  Inputs and weights are seeded, so two
builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the tree bench.py runs from may be read-only: nothing is cached in it

WORKLOADS = {
    # BASELINE.json configs[1]: 2x SR, seq_len=8, LR 128x128, batch=8 per GPU
    "cfg2": dict(scale=2, L=8, lr=(128, 128), B=8, desc="2x SR, seq_len=8, LR 128x128 synthetic events, batch=8/GPU"),
    # BASELINE.json configs[2]: 4x SR, seq_len=8, LR 128x128, batch=32 over 8 GPUs = 4 per GPU
    "cfg3": dict(scale=4, L=8, lr=(128, 128), B=4, desc="4x SR, seq_len=8, LR 128x128 synthetic events, batch=4/GPU"),
    # BASELINE.json configs[3]: 4x SR, seq_len=16, LR 256x256, batch=16 over 8 GPUs = 2 per GPU (long-sequence stress)
    "cfg4": dict(scale=4, L=16, lr=(256, 256), B=2, desc="4x SR, seq_len=16, LR 256x256 synthetic events, batch=2/GPU"),
}
EVENTS_PER_FRAME = 2048          # config/train_ours_enfssyn.yml:9 WINDOW
FLOP_PER_HR_PIXEL = 184.7e3      # SURVEY.md 8d
PARITY_TOL = 1e-3                # BASELINE.json north_star: within 1e-3 rel on fp32 count tensors
DUMP_BYTES = 60 << 20            # --dump-outputs: payload of all .npy files together (keeps the directory under 64 MB)


def synth_events(B, L, lr, seed):
    """SURVEY 8d synthetic input: n=2048 events per frame, x~U{0..W-1}, y~U{0..H-1}, p~U{-1,+1}."""
    g = torch.Generator().manual_seed(seed)
    n = B * L * EVENTS_PER_FRAME
    xs = torch.randint(0, lr[1], (n,), generator=g).float()
    ys = torch.randint(0, lr[0], (n,), generator=g).float()
    ps = (torch.randint(0, 2, (n,), generator=g) * 2 - 1).float()
    off = torch.arange(0, n + 1, EVENTS_PER_FRAME, dtype=torch.int64)
    return xs, ys, ps, off


def synth_weights(seed=0):
    """Random-init weights of the shipped architecture (fan-in scaled normal; non-zero conv_offset_mask so that the
    deformable sampling is exercised, BASELINE.md 3), keyed like the reference state_dict.  No checkpoint exists offline."""
    from esr_b200.model import DeepRecurrNet
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for k, v in DeepRecurrNet(inch=2, basech=8, num_frame=3).state_dict().items():
        shp = tuple(v.shape)
        if k.endswith(".weight"):
            fan_in = 1
            for d in shp[1:]:
                fan_in *= d
            std = 0.02 if "conv_offset_mask" in k else (1.0 / fan_in) ** 0.5
            sd[k] = torch.randn(shp, generator=g) * std
        else:
            sd[k] = torch.randn(shp, generator=g) * (0.3 if "conv_offset_mask" in k else 0.05)
    return sd


def synth_sr_bias(B, L, hr, seed):
    """A random-init network's output rounds to zero events (SURVEY 8d), so the redistribution stage is fed
    `model output + Poisson(0.3)` synthetic counts (BASELINE.md 3) to do representative work."""
    g = torch.Generator().manual_seed(seed + 17)
    return torch.poisson(torch.full(((L - 2) * B, 2, hr[0], hr[1]), 0.3), generator=g)


def dump_outputs(out_dir, arrays, budget=DUMP_BYTES):
    """Writes each tensor of `arrays` as out_dir/<name>.npy in float32.  When all of them together exceed `budget`, each one is
    replaced by a fixed sample of its flattened elements (seed 0, ascending index, a share of the budget proportional to its
    size): the same shapes give the same indices, so two builds run with the same arguments compare element for element."""
    os.makedirs(out_dir, exist_ok=True)
    total = sum(t.numel() for t in arrays.values()) * 4
    for name, t in arrays.items():
        a = t.detach().float()
        if total > budget:
            k = t.numel() * budget // total
            idx = np.unique(np.random.default_rng(0).integers(0, t.numel(), k))
            a = a.reshape(-1)[torch.from_numpy(idx).to(a.device)]
        np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy())


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons of ONE GPU during the timed region.  NVML in-process (nvidia_ml_py): a query costs
    microseconds; spawning `nvidia-smi` per sample from every rank (the first version) took the driver lock for ~0.5 s each
    and visibly slowed the timed steps at N >= 4.  Falls back to one nvidia-smi call per second if NVML is unavailable."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.stop_flag = gpu_index, [], False
        self.nvml, self.handle = None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            try:
                uuid = "GPU-" + str(torch.cuda.get_device_properties(gpu_index).uuid)
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(uuid)
            except Exception:
                vis = os.environ.get("CUDA_VISIBLE_DEVICES")
                idx = int(vis.split(",")[gpu_index]) if vis and vis.split(",")[gpu_index].isdigit() else gpu_index
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n, h = self.nvml, self.handle
        sm = n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM)
        try:
            bits = n.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:
            bits = n.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        flag = lambda m: "Active" if bits & m else "Not Active"
        # bit masks (nvml.h): SwPowerCap 0x4, HwSlowdown 0x8, SwThermalSlowdown 0x20, HwThermalSlowdown 0x40
        self.rows.append([str(self.gpu), str(sm), str(mx), "", hex(bits), flag(0x8), flag(0x40), flag(0x20), flag(0x4)])

    def run(self):
        while not self.stop_flag:
            try:
                if self.nvml is not None:
                    self._sample_nvml()
                else:
                    out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.gpu)],
                                         capture_output=True, text=True, timeout=5).stdout.strip()
                    if out:
                        self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.02 if self.nvml is not None else 1.0)

    def summary(self):
        sm = [float(r[1]) for r in self.rows if len(r) > 2 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def usable_cores(cap=32):
    """Host threads the CPU legs may use: affinity and cgroup quota, capped (torch's small convs stop scaling, and
    oversubscribing a 128-way box made the oracle ~100x slower when measured)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(per))))
    except Exception:
        pass
    return max(1, min(n, cap))


_JSON_OUT = sys.stdout


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1443.7), d.get("hbm_gbs", 6574.1), "measured (MEASURED_PEAKS.json)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(workload):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed summary of an
    `ncu --set full` capture (profiles/r2_ncu_traffic.json, written by tools/ncu_traffic.py with the capture's git hash).
    Nothing is hard-coded here: no file, or no entry for this workload -> None."""
    p = os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")
    try:
        d = json.load(open(p))
        e = d.get(workload)
        if e:
            return e
    except Exception:
        pass
    return None


# ------------------------------------------------------------------------------------------------------------------
# CPU legs (oracle port + the reference's own compiled Cython where it was built): test infrastructure used as baseline
# ------------------------------------------------------------------------------------------------------------------
_REF_C2E = "unset"


def reference_cnt2event():
    """The reference's own cnt2event Cython module compiled from /root/reference (oracle/_ref, built in the build container,
    shipped to the GPU box as a .so) or None."""
    global _REF_C2E
    if _REF_C2E == "unset":
        try:
            from oracle import build_ref
            _REF_C2E = build_ref.import_ref_modules()[0]
        except Exception:
            _REF_C2E = None
    return _REF_C2E


REF_C2E_EVENT_CAP = 4e5          # the reference's Cython runs at ~65 k events/s (SURVEY 8a row 15): bound what one pass feeds it


def cpu_oracle_step(wl, B_sample, sd, seed, use_ref_cython=True):
    """One step of the CPU path on a sample of B_sample sequences.  Returns (seconds, events, stage seconds, redistribution kind).
    With the reference's Cython the redistribution is run on the first SR frames holding <= REF_C2E_EVENT_CAP events and its
    time scaled linearly to all frames (cnt2event is a per-sample loop, linear in the event count; SURVEY 8d allows exactly this
    extrapolation) -- the kind string says when that happened."""
    from oracle import events as oe
    from oracle import model_ref
    scale, L, lr = wl["scale"], wl["L"], wl["lr"]
    hr = (lr[0] * scale, lr[1] * scale)
    xs, ys, ps, off = synth_events(B_sample, L, lr, seed)
    xs, ys, ps, off = xs.numpy(), ys.numpy(), ps.numpy(), off.numpy()
    bias = synth_sr_bias(B_sample, L, hr, seed)
    net = model_ref.OracleNet(sd)
    ref_c2e = reference_cnt2event() if use_ref_cython else None
    t0 = time.perf_counter()
    frames = np.empty((B_sample * L, 2, hr[0], hr[1]), np.float32)
    for f in range(B_sample * L):
        a, b = off[f], off[f + 1]
        frames[f] = oe.events_to_channels(oe.lift_coords(xs[a:b], lr[1], hr[1]), oe.lift_coords(ys[a:b], lr[0], hr[0]),
                                          ps[a:b], hr)
    t1 = time.perf_counter()
    bank = torch.from_numpy(frames).view(B_sample, L, 2, hr[0], hr[1])
    net.reset_states()
    outs = [net(bank[:, w:w + 3].contiguous()) for w in range(L - 2)]
    sr = torch.cat(outs, 0) + bias
    t2 = time.perf_counter()
    kind = "port"
    if ref_c2e is not None:
        arr = np.ascontiguousarray(sr.numpy(), dtype=np.float32)
        per_frame = np.rint(np.abs(arr)).reshape(arr.shape[0], -1).sum(1)
        k = int(max(1, min(arr.shape[0], np.searchsorted(np.cumsum(per_frame), REF_C2E_EVENT_CAP) + 1)))
        t2 = time.perf_counter()
        ev = ref_c2e.cnt2event(arr[:k], 0)                                                 # cnt2event.pyx:18-116, unmodified
        dt_r = (time.perf_counter() - t2) * float(per_frame.sum() / max(per_frame[:k].sum(), 1.0))
        n_ev = int(per_frame.sum())
        kind = "reference" if k == arr.shape[0] else f"reference ({k} of {arr.shape[0]} SR frames run, time scaled by event count)"
    else:
        ev = oe.cnt2event(sr.numpy(), 0)
        dt_r = time.perf_counter() - t2
        n_ev = int((ev[:, :, 3] != 0).sum())
    return (t2 - t0) + dt_r, n_ev, (t1 - t0, t2 - t1, dt_r), kind


def cpu_baseline_for(wl, sd, budget_s=12.0):
    """The CPU path on a bounded sample of the workload (about `budget_s` seconds of CPU work)."""
    cores = usable_cores()
    torch.set_num_threads(cores)
    L, B = wl["L"], wl["B"]
    t1, _, _, kind = cpu_oracle_step(wl, 1, sd, 1)                 # warm-up + sizing: one sequence
    b_s = int(min(B, max(1, round(budget_s / 3.0 / max(t1, 1e-3)))))
    ts, stages, spent = [], np.zeros(3), 0.0
    while spent < budget_s * 0.8 or len(ts) < 1:
        dt, _, st, kind = cpu_oracle_step(wl, b_s, sd, 1)
        ts.append(dt)
        stages += np.array(st)
        spent += dt
        if len(ts) >= 8:
            break
    tcpu = float(np.mean(ts))
    stages /= len(ts)
    # the same sample with the C port of cnt2event instead of the reference's Cython (its per-pixel numpy allocations and
    # Python sorted() are ~100x slower than a plain C loop; SURVEY 8a row 15): reported so that both readings are visible
    tport, _, stp, _ = cpu_oracle_step(wl, b_s, sd, 1, use_ref_cython=False)
    return {"value": b_s * L / tcpu, "unit": "frames/s", "cores": cores, "kind": "port",
            "sample": f"{b_s} sequence(s) x {L} LR frames per pass (the GPU arm's step is B={B}), mean of {len(ts)} passes = {spent:.1f} s of CPU work, fp32",
            "parts": {"encode": "C oracle (port)", "network": "torch fp32 oracle (port), %d threads" % cores,
                      "redistribute": ("reference's own Cython cnt2event (oracle/_ref): " + kind) if kind.startswith("reference") else "C oracle (port)"},
            "stage_s_per_pass": {"encode": float(stages[0]), "network": float(stages[1]), "redistribute": float(stages[2])},
            "value_with_c_port_redistribution": b_s * L / tport}


def cpu_oracle_train_step(wl, sd, seed):
    """One training iteration (windows with carried state, summed MSE, backward, torch Adam amsgrad) of the CPU oracle on
    ONE sequence.  Returns seconds."""
    import torch.nn.functional as F
    from oracle import model_ref
    scale, L, lr = wl["scale"], wl["L"], wl["lr"]
    H, W = lr[0] * scale, lr[1] * scale
    g = torch.Generator().manual_seed(seed)
    frames = torch.poisson(torch.full((1, L, 2, H, W), 0.1), generator=g)
    gt = torch.poisson(torch.full((1, L, 2, H, W), 0.1), generator=g)
    params = {k: v.clone().requires_grad_() for k, v in sd.items()}
    opt = torch.optim.Adam(list(params.values()), lr=1e-3, weight_decay=1e-4, amsgrad=True)
    t0 = time.perf_counter()
    opt.zero_grad()
    states, loss = None, 0
    for w in range(L - 2):
        pred, states = model_ref.forward(params, frames[:, w:w + 3], states)
        loss = loss + F.mse_loss(pred, gt[:, w + 1])
    loss.backward()
    opt.step()
    return time.perf_counter() - t0


def run_reference(args, wl, rank, world):
    if rank != 0:
        return
    cores = usable_cores()
    torch.set_num_threads(cores)
    sd = synth_weights(0)
    # each step = a bounded sample of the workload: as many sequences as take ~3 s on this host (at most the GPU arm's batch);
    # the whole run is held under ~3 minutes (K is honoured unless that bound would be exceeded)
    t1, _, _, kind = cpu_oracle_step(wl, 1, sd, 1)
    B_sample = int(min(wl["B"], max(1, round(3.0 / max(t1, 1e-3)))))
    for _ in range(max(0, min(args.warmup, 2) - 1)):
        cpu_oracle_step(wl, B_sample, sd, 1)
    times, budget = [], 170.0 - t1
    for _ in range(max(1, args.steps)):
        times.append(cpu_oracle_step(wl, B_sample, sd, 1)[0])
        budget -= times[-1]
        if budget < times[-1]:
            break
    t = float(np.mean(times))
    val = B_sample * wl["L"] / t
    redis = ("the reference's own Cython cnt2event (oracle/_ref, compiled unmodified): " + kind) if kind.startswith("reference") else "C oracle port"
    sample = (f"{B_sample} sequence(s) x {wl['L']} LR frames per step (B={wl['B']} in the GPU arm), {len(times)} steps, fp32: "
              f"C oracle encode + torch CPU oracle network ({cores} threads) + {redis}")
    line = {"impl": "reference", "metric": "LR event-frames/sec", "value": val, "unit": "frames/s", "n_gpus": args.gpus,
            "steps": len(times), "warmup": min(args.warmup, 2), "ms_per_step": t * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": {"workload": wl["desc"], "impl_note": "CPU restatement of the reference path (oracle/): the reference's own "
                       "Python network cannot travel to the GPU box; its compiled Cython redistribution can and is used when present"},
            "cpu_baseline": {"value": val, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample,
                             "redistribute_kind": kind},
            "e2e": {"value": val, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    _JSON_OUT.write(json.dumps(line) + "\n")
    _JSON_OUT.flush()


# ------------------------------------------------------------------------------------------------------------------
# GPU legs
# ------------------------------------------------------------------------------------------------------------------
def measure_training(args, wl, net_sd, dev, rank, world, dist, steps=None, cpu=True):
    """SURVEY 8a row 17 / 8d: the training iteration (forward of all windows, backward through time, gradient all-reduce
    when N > 1, Adam amsgrad) on the same workload, replayed from ONE CUDA graph (at N > 1 the NCCL all-reduce of the flat
    1.8 M-element gradient is captured inside it; falls back to eager launches if the capture is refused).
    Device-resident synthetic count tensors (the trainer's input after the dataloader)."""
    from esr_b200 import train
    from esr_b200.model import DeepRecurrNet
    scale, L, lr, B = wl["scale"], wl["L"], wl["lr"], wl["B"]
    H, W = lr[0] * scale, lr[1] * scale
    net = DeepRecurrNet(inch=2, basech=8, num_frame=3)
    net.load_state_dict(net_sd)
    net = net.to(dev)
    opt = train.Adam(net.parameters(), lr=1e-3, weight_decay=1e-4, amsgrad=True)
    g = torch.Generator().manual_seed(200 + rank)
    frames = torch.poisson(torch.full((B, L, 2, H, W), 0.1), generator=g).to(dev)
    gt = torch.poisson(torch.full((B, L, 2, H, W), 0.1), generator=g).to(dev)
    mode, allred, grad_check = "one CUDA graph per iteration", None, None
    if world > 1:
        def allred(flat):
            dist.all_reduce(flat, op=dist.ReduceOp.AVG)
    step = None
    if not args.no_graph:
        try:
            gstep = train.GraphedTrainStep(net, opt, tuple(frames.shape), dev, all_reduce=allred)
            step = lambda: gstep(frames, gt)
            if world > 1:
                mode = "one CUDA graph per iteration incl. the NCCL all-reduce of the flat gradient"
        except Exception as e:                                         # capture refused (NCCL / allocator): run eagerly, say so
            sys.stderr.write(f"[bench] graph capture of the training iteration failed, running eagerly: {e}\n")
            torch.cuda.synchronize()
            step = None
    ok = torch.tensor([1.0 if step is not None else 0.0], device=dev)
    if world > 1:
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if ok.item() == 0.0:
        step = lambda: train.train_step(net, opt, frames, gt, all_reduce=allred)
        mode = "eager" + (" + NCCL all-reduce of the flat gradient" if world > 1 else "")
    steps = steps or max(3, min(args.steps, 10))
    for _ in range(3):
        step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    first = last = None
    for i in range(steps):
        l = step()
        if i == 0:
            first = l.clone()
        last = l
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = t.item() / steps
    if world > 1:                                                     # after the timed loop: an eager backward on the default
        #                                                               stream before the capture invalidated it (measured at N = 2)
        # gradient-exchange check on hardware (pytest -m gpu has one GPU): after the all-reduce every rank must hold the same
        # flat gradient, equal to the mean of the per-rank gradients gathered separately
        opt.zero_grad()
        net.reset_states()
        pred = net(frames)
        Wn = L - 2
        loss = Wn * train.mse_loss(pred, gt[:, 1:1 + Wn].transpose(0, 1).reshape(pred.shape))
        loss.backward()
        opt.log[0] = float(rank + 1)                                  # the logging slots ride in the same bucket
        opt.log[1] = loss.detach()
        local = opt.exchange.clone()
        gathered = [torch.empty_like(local) for _ in range(world)]
        dist.all_gather(gathered, local)
        want = torch.stack(gathered).mean(0)
        allred(opt.exchange)
        err = ((opt.exchange - want).abs().max() / want.abs().max().clamp_min(1e-30)).item()
        same = torch.tensor([float(opt.exchange.double().sum())], dtype=torch.float64, device=dev)
        lo, hi = same.clone(), same.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        log_ok = abs(float(opt.log[0]) - (world + 1) / 2.0) < 1e-5
        grad_check = {"rel_err_vs_mean_of_gathered": err, "identical_on_all_ranks": bool((hi - lo).abs().item() == 0.0),
                      "logging_scalars_reduced_in_the_same_bucket": bool(log_ok),
                      "ok": bool(err < 1e-5 and (hi - lo).abs().item() == 0.0 and log_ok)}
        opt.zero_grad()
    out = {"metric": "training LR event-frames/sec (forward + backward + Adam)", "value": world * B * L / (ms * 1e-3), "unit": "frames/s",
           "ms_per_step": ms, "steps": steps, "mode": mode,
           "batch_per_gpu": B, "loss_first": float(first), "loss_last": float(last),
           "peak_mem_gb": torch.cuda.max_memory_allocated() / 2 ** 30}
    if grad_check is not None:
        out["gradient_exchange_check"] = grad_check
    if rank == 0 and world == 1 and cpu and not args.no_cpu_baseline:
        cores = usable_cores()
        torch.set_num_threads(cores)
        tcpu = cpu_oracle_train_step(wl, net_sd, 3)
        out["cpu_baseline"] = {"value": L / tcpu, "unit": "frames/s", "cores": cores, "kind": "port",
                               "sample": f"1 sequence x {L} LR frames, one iteration, torch CPU autograd through the oracle + torch Adam"}
    del net, opt
    return out


def parity_check(net, pipe, wl, sd, n_seq):
    """Un-timed: the network output of the plan bench.py measures (full batch B, all windows, state carried) against the CPU
    oracle on the first n_seq sequences of the very same input bank.  Returns the `parity` object of the JSON line."""
    from oracle import model_ref
    scale, L, lr, B = wl["scale"], wl["L"], wl["lr"], wl["B"]
    H, W = lr[0] * scale, lr[1] * scale
    torch.set_num_threads(usable_cores())
    t0 = time.perf_counter()
    with torch.no_grad():
        net.reset_states()
        frames = pipe.bank.view(B, L, 2, H, W)
        got = net.forward_sequence(frames).view(L - 2, B, 2, H, W)[:, :n_seq].cpu()
        st = [s[:n_seq].cpu() for s in net.states(B, L, H, W)]
        host = frames[:n_seq].cpu()
    ora = model_ref.OracleNet(sd)
    rel = lambda a, b: ((a - b).abs().max() / b.abs().max().clamp_min(1e-12)).item()
    per_window = []
    for w in range(L - 2):
        per_window.append(rel(got[w], ora(host[:, w:w + 3].contiguous())))
    st_rel = [rel(a, b) for a, b in zip(st, ora.states)]
    worst = max(per_window + st_rel)
    return {"rel_max": worst, "tolerance": PARITY_TOL, "ok": bool(worst < PARITY_TOL), "per_window_rel": per_window,
            "carried_state_rel": st_rel, "windows": L - 2, "sequences_checked": n_seq, "batch": B,
            "oracle": "oracle/model_ref.py (fp32 torch CPU restatement, pinned to the reference's own outputs by tests/golden/model_golden.npz)",
            "norm": "max |got - want| / max |want| per window output and per carried state", "seconds": time.perf_counter() - t0}


def profile_launches(net, wl, dev, reps=5):
    """Per-launch CUDA-event timing of one sequence batch through esr_net_forward_profiled: [(name, class, ms, flops, bytes)]."""
    import ctypes
    from esr_b200 import _lib
    scale, L, lr, B = wl["scale"], wl["L"], wl["lr"], wl["B"]
    hr = (lr[0] * scale, lr[1] * scale)
    plan = net._plans[(B, L, hr[0], hr[1])]
    bank = torch.poisson(torch.full((B * L, 2, hr[0], hr[1]), 0.1)).to(dev)
    out = torch.empty(((L - 2) * B, 2, hr[0], hr[1]), device=dev)
    cap = 256
    cls, ms, fl, by = (ctypes.c_int * cap)(), (ctypes.c_float * cap)(), (ctypes.c_double * cap)(), (ctypes.c_double * cap)()
    names = ctypes.create_string_buffer(32 * cap)
    cnt = ctypes.c_int(0)
    acc = None
    for r in range(reps + 1):
        _lib.check(_lib.lib().esr_net_forward_profiled(plan.handle, _lib.ptr(bank), None, _lib.ptr(out), cap, ctypes.byref(cnt),
                                                       cls, ms, fl, by, names, _lib.stream_ptr()), "profiled forward")
        if r == 0:
            continue                                                 # warm-up
        if acc is None:
            acc = [[names.raw[32 * i:32 * i + 32].split(b"\0")[0].decode(), int(cls[i]), 0.0, float(fl[i]), float(by[i])]
                   for i in range(cnt.value)]
        for i in range(cnt.value):
            acc[i][2] += ms[i] / reps
    return [tuple(a) for a in acc]


def rooflines(rows, wl_name, peak_tf, peak_hbm, peak_src):
    """roofline (tensor, dominant family) + the HBM-bound small-channel convs from the per-launch table."""
    tc = [r for r in rows if r[1] == 0]
    gru = [r for r in rows if r[1] == 3]
    direct = [r for r in rows if r[1] == 1]
    other = [r for r in rows if r[1] == 2]
    tot_ms = sum(r[2] for r in rows)
    fam_fl, fam_ms = sum(r[3] for r in tc), sum(r[2] for r in tc)
    fam_tf = fam_fl / (fam_ms * 1e-3) / 1e12 if fam_ms else 0.0
    all_fl, all_ms = fam_fl + sum(r[3] for r in gru), fam_ms + sum(r[2] for r in gru)
    all_tf = all_fl / (all_ms * 1e-3) / 1e12 if all_ms else 0.0
    best = max(tc, key=lambda r: r[3] / max(r[2], 1e-9), default=None)
    top = max(tc, key=lambda r: r[3], default=None)
    tf = lambda r: r[3] / (r[2] * 1e-3) / 1e12 if r and r[2] > 0 else 0.0
    traffic = ncu_traffic(wl_name)
    roof = {"kernel": "k_conv_tc / k_conv_tc_persist family (tcgen05 implicit-GEMM convs): every tensor-core conv launch of one step, FLOP-weighted",
            "bound": "tensor", "achieved": fam_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": fam_tf / peak_tf,
            "peak_source": peak_src + ", bf16 sustained",
            "algorithmic_gflop_per_step": fam_fl / 1e9, "ms_per_step": fam_ms, "launches_per_step": len(tc),
            "share_of_step_kernel_time": fam_ms / tot_ms if tot_ms else None,
            "note": "algorithmic FLOPs (1x); the fp32-parity 3-pass split-bf16 product issues 3x that on the tensor pipe, so 1/3 is this family's ceiling",
            "traffic": traffic["dram_bytes_per_launch"] if traffic else None, "traffic_source": traffic,
            "largest_launch": {"layer": top[0], "achieved": tf(top), "frac": tf(top) / peak_tf, "launch_ms": top[2],
                               "algorithmic_gflop": top[3] / 1e9} if top else None,
            "best_launch": {"layer": best[0], "achieved": tf(best), "frac": tf(best) / peak_tf, "launch_ms": best[2]} if best else None,
            "with_gru_chain": {"achieved": all_tf, "frac": all_tf / peak_tf, "gru_chain_ms_per_step": sum(r[2] for r in gru),
                               "gru_chain_tflops": tf(gru[0]) if gru else None},
            "per_layer": [{"layer": r[0], "ms": round(r[2], 5), "tflops": round(tf(r), 1)} for r in tc]}
    d_by, d_ms = sum(r[4] for r in direct), sum(r[2] for r in direct)
    small = {"kernel": "k_conv_mma<...> small-channel full-resolution convs (head+enc0, enc1, enc2, attention maps, recons[1,2], tail), byte-weighted",
             "bound": "hbm", "achieved": d_by / (d_ms * 1e-3) / 1e9 if d_ms else 0.0, "peak": peak_hbm, "unit": "GB/s",
             "frac": d_by / (d_ms * 1e-3) / 1e9 / peak_hbm if d_ms else 0.0, "ms_per_step": d_ms, "algorithmic_mb_per_step": d_by / 1e6,
             "traffic": None,
             "per_layer": [{"layer": r[0], "ms": round(r[2], 5), "GBps": round(r[4] / (r[2] * 1e-3) / 1e9, 1) if r[2] > 0 else None}
                           for r in direct]}
    ew = {"ms_per_step": sum(r[2] for r in other), "algorithmic_mb_per_step": sum(r[4] for r in other) / 1e6,
          "per_layer": [{"layer": r[0], "ms": round(r[2], 5), "GBps": round(r[4] / (r[2] * 1e-3) / 1e9, 1) if r[2] > 0 else None}
                        for r in other]}
    return roof, small, ew


def run_workload(args, name, dev, rank, world, dist, steps, warmup, main):
    """Times one network workload on this rank's shard.  main=True adds the one-at-a-time e2e view, the stage breakdown,
    the per-launch rooflines and the clock record."""
    from esr_b200 import _lib
    from esr_b200 import encodings as enc
    from esr_b200.expand import expand
    from esr_b200.model import DeepRecurrNet
    from esr_b200.pipeline import EventSRPipeline
    wl = WORKLOADS[name]
    scale, L, lr, B = wl["scale"], wl["L"], wl["lr"], wl["B"]
    hr = (lr[0] * scale, lr[1] * scale)
    sd = synth_weights(0)
    net = DeepRecurrNet(inch=2, basech=8, num_frame=3)
    net.load_state_dict(sd)
    net = net.to(dev).eval()
    pipe = EventSRPipeline(net, B, L, lr, scale, dev)
    pipe.sr_bias = synth_sr_bias(B, L, hr, 100 + rank).to(dev)
    xs, ys, ps, off = synth_events(B, L, lr, 100 + rank)
    h_xs, h_ys, h_ps, h_off = (t.pin_memory() for t in (xs, ys, ps, off))
    d_xs, d_ys, d_ps, d_off = (t.to(dev) for t in (xs, ys, ps, off))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        """per-step CUDA-event timing with an (untimed) L2 flush between steps; returns (total ms, what the last step returned)"""
        tot, out = 0.0, None
        for _ in range(k):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            out = fn()
            e1.record()
            torch.cuda.synchronize()
            tot += e0.elapsed_time(e1)
        return tot, out

    dev_step = lambda: pipe.run_device(d_xs, d_ys, d_ps, d_off, EVENTS_PER_FRAME)
    host_step = lambda: pipe.run_host(h_xs, h_ys, h_ps, h_off, EVENTS_PER_FRAME)

    dev_step()
    if not args.no_graph:
        pipe.capture()
    for _ in range(warmup):
        dev_step()
        host_step()
        pipe.collect(pipe.submit_host(h_xs, h_ys, h_ps, h_off, EVENTS_PER_FRAME))
    sampler = ClockSampler(dev.index if dev.index is not None else 0) if main else None
    if sampler:
        sampler.start()
    barrier()
    l0 = _lib.lib().esr_launch_count()
    ms_dev, last = timed(dev_step, steps)
    launches = _lib.lib().esr_launch_count() - l0 + steps * pipe.graph_launches
    if main and rank == 0 and args.dump_outputs:                      # before the next step overwrites the graph's output buffers
        dump_outputs(args.dump_outputs, {"sr_counts": last[0], "events": last[1]})
    del last
    barrier()
    ms_e2e_sync = timed(host_step, steps)[0] if main else 0.0         # one batch at a time (latency view)
    barrier()

    # throughput view of the same end-to-end path: submit(i+1) is issued before finish(i), so the GPU runs batch i+1's network while
    # the host waits for / sizes batch i's event list, and the D2H of batch i-1 drains on a side stream (three in flight).
    # One timed region around all K steps (inputs + workspace exceed L2; no flush inside, it would serialise the overlap).
    def pipelined(k):
        pend_a, pend_b = None, None                # submitted (network queued) / finished (D2H in flight)
        for _ in range(k):
            h = pipe.submit_host(h_xs, h_ys, h_ps, h_off, EVENTS_PER_FRAME)
            if pend_a is not None:
                hb = pipe.finish(pend_a)            # host sizes batch i-1's output while the GPU runs batch i's network
                if pend_b is not None:
                    pipe.collect(pend_b)
                pend_b = hb
            pend_a = h
        for hdl in (pend_b, pend_a):
            if hdl is not None:
                pipe.collect(hdl)

    # warm-up of THIS loop form: with three batches in flight the caching allocator needs one more set of event / workspace
    # blocks than the one-at-a-time form; their first cudaMalloc synchronises the device and would land in the timed region
    pipelined(max(warmup, 3) + 1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    flush.zero_()
    torch.cuda.synchronize()
    e0.record()
    pipelined(steps)
    e1.record()
    torch.cuda.synchronize()
    ms_e2e = e0.elapsed_time(e1)
    barrier()
    clocks = None
    if sampler:
        sampler.stop_flag = True
        sampler.join(timeout=2)
        clocks = sampler.summary()

    t = torch.tensor([ms_dev, ms_e2e, ms_e2e_sync], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_dev, ms_e2e, ms_e2e_sync = t.tolist()
    frames_per_step = world * B * L
    res = {"workload": wl["desc"], "value": frames_per_step * steps / (ms_dev / 1e3), "unit": "frames/s", "steps": steps,
           "ms_per_step": ms_dev / steps, "batch_per_gpu": B,
           "sr_frames_per_s": frames_per_step * steps / (ms_dev / 1e3) * (L - 2) / L}
    n_ev = EVENTS_PER_FRAME * B * L
    ev_out = dev_step()[1]
    res["e2e"] = {"value": frames_per_step * steps / (ms_e2e / 1e3), "unit": "frames/s", "ms_per_step": ms_e2e / steps,
                  "mode": "software-pipelined, three batches in flight: H2D + step graph (encode input -> network -> redistribution) of batch i+1 | host reads batch i's size | D2H of batch i's event list on a side stream",
                  "h2d_bytes_per_step": int(n_ev * 12 + (B * L + 1) * 8), "d2h_bytes_per_step": int(ev_out.numel() * 4)}
    if main:
        res["e2e"]["one_at_a_time"] = {"value": frames_per_step * steps / (ms_e2e_sync / 1e3), "ms_per_step": ms_e2e_sync / steps}
    res["gpu_launches"] = int(launches)
    res["clocks"] = clocks
    res["whole_path_algorithmic_tflops"] = FLOP_PER_HR_PIXEL * hr[0] * hr[1] * B * (L - 2) * world / (ms_dev / steps / 1e3) / 1e12

    if rank == 0:
        peak_tf, peak_hbm, peak_src = measured_peaks()
        # ---- parity of the measured plan against the oracle (un-timed)
        if not args.no_parity:
            res["parity"] = parity_check(net, pipe, wl, sd, n_seq=min(B, 2 if name == "cfg2" else 1))
        # ---- per-launch rooflines (live CUDA events)
        rows = profile_launches(net, wl, dev)
        roof, small, ew = rooflines(rows, name, peak_tf, peak_hbm, peak_src)
        res["roofline"] = roof
        res["_small"], res["_ew"], res["_rows"] = small, ew, rows
        # ---- stage breakdown of one step (device-resident inputs), CUDA events on the launching stream.  With graphs the
        # redistribution is part of the replay: it is timed as its own small graph (same kernels, memsets and statistics copy) on
        # the SR counts of this step, and the network is the replay minus that.
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        acc3 = [0.0, 0.0, 0.0]
        reps = 5
        rd_graph = None
        if pipe._graph is not None:
            from esr_b200.expand import FusedCnt2Event
            f0 = pipe._graphs[0]["fused"]
            fz = FusedCnt2Event(f0.B, f0.H, f0.W, dev, f0.cap, f0.mcap)
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                fz.enqueue(pipe._graph_sr)
            torch.cuda.current_stream().wait_stream(side)
            rd_graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(rd_graph):
                fz.enqueue(pipe._graph_sr)
        for _ in range(reps):
            flush.zero_()
            torch.cuda.synchronize()
            ev[0].record()
            with torch.no_grad():
                enc.encode_frames(d_xs, d_ys, d_ps, d_off, lr_size=lr, hr_size=hr, n_max_frame=EVENTS_PER_FRAME, out=pipe.bank)
            ev[1].record()
            with torch.no_grad():
                if pipe._graph is not None:
                    pipe._graph.replay()
                    sr_ = pipe._graph_sr
                else:
                    sr_ = pipe._windows()
            ev[2].record()
            if rd_graph is not None:
                torch.cuda.synchronize()
                flush.zero_()
                torch.cuda.synchronize()
                ev[3].record()
                rd_graph.replay()
                ev[4].record()
                torch.cuda.synchronize()
                evs = fz.result()[0]
                rd = ev[3].elapsed_time(ev[4])
                acc3[0] += ev[0].elapsed_time(ev[1]) / reps
                acc3[1] += (ev[1].elapsed_time(ev[2]) - rd) / reps
                acc3[2] += rd / reps
            else:
                evs = expand(sr_, 0, 0)
                ev[3].record()
                torch.cuda.synchronize()
                for i in range(3):
                    acc3[i] += ev[i].elapsed_time(ev[i + 1]) / reps
        res["stages_ms_per_step"] = {"encode_ms": acc3[0], "network_ms": acc3[1], "redistribute_ms": acc3[2]}
        # HBM-bound stages against the measured copy bandwidth: SURVEY 8d algorithmic bytes
        nfr, nout = B * L, B * (L - 2)
        E = int((evs[:, :, 3] != 0).sum().item())
        b_sc = 12.0 * n_ev + 8.0 * hr[0] * hr[1] * nfr
        b_rd = 8.0 * hr[0] * hr[1] * nout + 16.0 * E
        hbm = lambda b, ms_: {"bound": "hbm", "achieved": b / (ms_ * 1e-3) / 1e9, "peak": peak_hbm, "unit": "GB/s",
                              "frac": b / (ms_ * 1e-3) / 1e9 / peak_hbm, "ms_per_step": ms_, "algorithmic_mb_per_step": b / 1e6, "traffic": None}
        res["roofline_hbm"] = {
            "scatter": dict(hbm(b_sc, acc3[0]), kernel="k_scatter_cnt (LR->HR lift + count scatter of all B*L frames, one launch)",
                            bytes="12 B per event + 8*H*W per frame (SURVEY 8d)", events=n_ev),
            "redistribute": dict(hbm(b_rd, acc3[2]), kernel="k_xf_count -> k_xf_scan -> k_xf_emit (csrc/expand_fused.cu: counting sort over the distinct timestamps, sized on the "
                                        "device, part of the step's CUDA graph); general chain of events.cu when a count exceeds 64",
                                 bytes="8*H*W per sample + 16 B per event (SURVEY 8d)", events=E),
            "small_convs": small, "elementwise": ew, "peak_source": peak_src + ", copy bandwidth"}
    del pipe, net, flush
    torch.cuda.empty_cache()
    return res, sd


def sweep_events(dev, peak_hbm, cpu=True):
    """BASELINE.json configs[4]: count scatter + redistribution at 1e5 .. 1e7 events per chunk on a 256x256 grid, achieved GB/s
    against the measured HBM peak, with the CPU column (torch index_put_ as in dataloader/encodings.py:243-268 for the scatter;
    the reference's own Cython cnt2event for the redistribution, bounded to <= 2e5 events and extrapolated linearly)."""
    from esr_b200 import encodings as enc
    from esr_b200.expand import expand
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def timed(fn, reps=5):
        fn()
        ts = []
        for _ in range(reps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return sorted(ts)[len(ts) // 2]

    H = 256
    g = torch.Generator(device=dev).manual_seed(1)
    pts = []
    for n in (10 ** 5, 10 ** 6, 10 ** 7):
        xs = torch.randint(0, H, (n,), generator=g, device=dev).float()
        ys = torch.randint(0, H, (n,), generator=g, device=dev).float()
        ps = (torch.randint(0, 2, (n,), generator=g, device=dev) * 2 - 1).float()
        off = torch.tensor([0, n], dtype=torch.int64, device=dev)
        ms = timed(lambda: enc.encode_frames(xs, ys, ps, off, hr_size=(H, H), n_max_frame=n))
        b = 12.0 * n + 8.0 * H * H
        p = {"op": "scatter_cnt", "grid": H, "events": n, "ms": ms, "GBps": b / ms / 1e6, "frac_hbm": b / ms / 1e6 / peak_hbm,
             "Mev_per_s": n / ms / 1e3}
        if cpu and n <= 10 ** 6:
            cx, cy, cp = xs.cpu(), ys.cpu(), ps.cpu()
            t0 = time.perf_counter()
            for pol in (1.0, -1.0):                                   # events_to_channels = two events_to_image calls
                img = torch.zeros((H, H))
                img.index_put_((cy.long(), cx.long()), cp * (cp * pol > 0).float() * cp, accumulate=True)
            p["cpu_Mev_per_s"] = n / (time.perf_counter() - t0) / 1e6
            p["cpu_kind"] = "torch CPU index_put_ (the reference's own operator, dataloader/encodings.py:266)"
        pts.append(p)
        del xs, ys, ps
    ref_c2e = reference_cnt2event() if cpu else None
    for E in (10 ** 5, 10 ** 6, 10 ** 7):
        lam = E / (2.0 * H * H)
        cnt = torch.poisson(torch.full((1, 2, H, H), lam, device=dev), generator=g)
        Et = int(cnt.sum().item())
        api_ms = timed(lambda: expand(cnt, 0, 0), reps=3)              # the call a user makes: kernels + host sizing + one sync
        ms, how = api_ms, "expand() call (general chain of events.cu: a count above 64)"
        mxc = int(cnt.max().item())
        if mxc <= 64:                                                   # as inside the pipeline: recorded once, replayed
            from esr_b200.expand import FusedCnt2Event
            fz = FusedCnt2Event(1, H, H, dev, int(Et * 1.25) + 4096, 2 * mxc)
            fz.enqueue(cnt)
            torch.cuda.synchronize()
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr):
                fz.enqueue(cnt)
            ms, how = timed(gr.replay, reps=5), "CUDA-graph replay of esr_cnt2event_fused (as in the pipeline's step graph)"
            assert fz.result()[0] is not None
        b = 8.0 * H * H + 16.0 * Et
        p = {"op": "cnt2event", "grid": H, "events": Et, "ms": ms, "GBps": b / ms / 1e6, "frac_hbm": b / ms / 1e6 / peak_hbm,
             "Mev_per_s": Et / ms / 1e3, "timed": how, "api_call_ms": api_ms, "max_count": mxc}
        if ref_c2e is not None and E == 10 ** 5:
            c = np.ascontiguousarray(cnt.cpu().numpy(), dtype=np.float32)
            t0 = time.perf_counter()
            ref_c2e.cnt2event(c, 0)
            p["cpu_Mev_per_s"] = Et / (time.perf_counter() - t0) / 1e6
            p["cpu_kind"] = "reference Cython cnt2event (oracle/_ref), measured at this point only; it is linear in the event count"
        pts.append(p)
        del cnt
    return pts


# ------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from the host instead of replaying a CUDA graph")
    ap.add_argument("--profile-out", default=None, help="write the per-launch timing table of one step here")
    ap.add_argument("--no-train", action="store_true", help="skip the training-iteration measurement (the `train` key)")
    ap.add_argument("--no-parity", action="store_true", help="skip the un-timed oracle check of the measured plan")
    ap.add_argument("--no-extra", action="store_true", help="skip the other configs (cfg3 / cfg4) and the cfg5 sweep")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the last timed step returned (SR count tensors, event lists) as DIR/<name>.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    # stdout carries exactly ONE line (the JSON): anything a library prints there (NCCL's version banner at N > 1) goes to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    global _JSON_OUT
    _JSON_OUT = os.fdopen(json_fd, "w")
    wl = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    if args.impl == "reference":
        run_reference(args, wl, rank, world)
        return

    import torch.distributed as dist

    assert torch.cuda.is_available(), "bench.py --impl ours needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # NCCL's version banner / debug lines must not share stdout with the JSON line
        dist.init_process_group("nccl", device_id=dev)

    res, sd = run_workload(args, args.workload, dev, rank, world, dist, args.steps, args.warmup, main=True)

    # ---- CPU baseline on rank 0, N=1 only
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_baseline = cpu_baseline_for(wl, sd, budget_s=14.0)

    # ---- training iteration (SURVEY 8a row 17): reported next to the inference headline, never mixed into `value`
    train_res = None
    if not args.no_train:
        train_res = measure_training(args, wl, sd, dev, rank, world, dist)

    # ---- the other BASELINE.json configs: 4x SR (cfg3) and the long-sequence 4x stress (cfg4), each on this rank's shard
    configs, sweep = {}, None
    if not args.no_extra:
        for name in ("cfg2", "cfg3", "cfg4"):
            if name == args.workload:
                continue
            k = max(3, min(args.steps, 10 if name != "cfg4" else 5))
            r, sd_x = run_workload(args, name, dev, rank, world, dist, k, 3, main=False)
            if rank == 0:
                for key in ("_small", "_ew", "_rows"):
                    r.pop(key, None)
                if "roofline" in r:
                    r["roofline"].pop("per_layer", None)
                if world == 1 and not args.no_cpu_baseline:
                    r["cpu_baseline"] = cpu_baseline_for(WORKLOADS[name], sd_x, budget_s=8.0)
            if not args.no_train:
                r["train"] = measure_training(args, WORKLOADS[name], sd_x, dev, rank, world, dist, steps=3, cpu=False)
            configs[name] = r
        if rank == 0:
            sweep = sweep_events(dev, measured_peaks()[1], cpu=(world == 1 and not args.no_cpu_baseline))

    if rank == 0:
        scale, L, lr, B = wl["scale"], wl["L"], wl["lr"], wl["B"]
        rows = res.pop("_rows", [])
        res.pop("_small", None)
        res.pop("_ew", None)
        if args.profile_out:
            with open(args.profile_out, "w") as f:
                f.write("idx,layer,class(0=tc,1=small-channel conv,2=other,3=gru_chain),ms,algorithmic_flops,algorithmic_bytes\n")
                for i, r in enumerate(rows):
                    f.write("%d,%s,%d,%.5f,%.0f,%.0f\n" % (i, r[0], r[1], r[2], r[3], r[4]))
        line = {"metric": "LR event-frames/sec", "value": res["value"], "unit": "frames/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "bf16x3 (split-bf16 tensor-core operands, fp32 accumulate) / fp32 elsewhere",
                "data": "synthetic",
                "config": {"workload": wl["desc"], "scale": scale, "seq_len": L, "lr": list(lr), "batch_per_gpu": B,
                           "events_per_frame": EVENTS_PER_FRAME, "windows_per_sequence": L - 2,
                           "redistribute_input": "model output + Poisson(0.3) synthetic counts",
                           "l2": "256 MiB buffer rewritten between timed steps (outside the timed intervals)",
                           "parallelism": f"dp{world} (batch shards, no data-path collective)",
                           "cuda_graph": not args.no_graph,
                           "plan": "sequence plan: per-frame and state-independent layers batched over all windows, ConvGRU chain serial"},
                "sr_frames_per_s": res["sr_frames_per_s"],
                "clocks": res["clocks"],
                "e2e": res["e2e"],
                "gpu_launches": res["gpu_launches"],
                "parity": res.get("parity"),
                "tensor_roofline_whole_path": {"algorithmic_tflops": res["whole_path_algorithmic_tflops"]},
                "stages_ms_per_step": res.get("stages_ms_per_step"),
                "train": train_res,
                "roofline": res.get("roofline"), "roofline_hbm": res.get("roofline_hbm"),
                "cpu_baseline": cpu_baseline,
                "configs": configs, "sweep": sweep}
        _JSON_OUT.write(json.dumps(line) + "\n")
        _JSON_OUT.flush()
    if world > 1:
        dist.barrier()                                                # rank 0's un-timed extras (parity, sweep, CPU legs) end before teardown
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
