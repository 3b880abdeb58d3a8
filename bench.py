#!/usr/bin/env python
"""Benchmark of the RNN-T joint + transducer-loss hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One "step" = one fused joint+loss forward AND backward over one synthetic batch.
  N = 1: B=32, T=400, U=100, H=1024, V=1024 -- BASELINE.json configs[1], the configuration the metric is quoted on.
  N > 1 (launched by torchrun, one rank per GPU): BASELINE.json configs[2] -- a GLOBAL batch of 256 utterances sharded
         by utterance (256/N per GPU, one launch per rank, no data-path collective; strong scaling); the weight
         gradients land directly in one flat bucket and their NCCL all-reduce (joint 1,049,600 + predictor
         3,150,848 fp32) starts as soon as dW/db are final, overlapping the activation-gradient GEMM.
         `--global-batch 0` selects the round-1 weak-scaling workload (B=32 per GPU) instead.
The encoder features are handed over as the reference does (rnnt/model.py:27-28): a (B,T,H) VIEW of a (B,H,T) tensor.
Rank 0 prints ONE JSON line.

`--impl reference` times the reference's own CPU implementation of the path (torch nn.functional.linear + tanh +
torchaudio.functional.rnnt_loss forward+backward, i.e. rnnt/joint.py:25-39 + rnnt/model.py:35-41 restated in
oracle/ref_path.py) on the box's host cores, on BASELINE.json configs[0] (B=4,T=200,U=40), the reference's own
CPU-runnable case.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "RNN-T joint+loss fwd+bwd lattice-cells/s at B=32,T=400,U=100,V=1024"
UNIT = "lattice-cells/s"
B, T, U, H, V = 32, 400, 100, 1024, 1024
PRED_GRAD_ELEMS = 3_150_848        # ConvPredictor parameters (SURVEY 2.1) that ride the same all-reduce
FLOP_PER_CELL_GEMM = 2 * H * V     # one H x V contraction per lattice cell
CPU_SAMPLE = dict(B=4, T=200, U=40)   # BASELINE.json configs[0] / BASELINE.md section 4
GLOBAL_BATCH = 256                    # BASELINE.json configs[2]


def load_peaks():
    """Roofline denominators: MEASURED_PEAKS.json (driver-written) -- burst for short timed regions, sustained for
    seconds-long loops under the power cap -- else the fallback B200_PROFILING.md states."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        burst = float(p.get("bf16_tflops", 1590.0))
        return dict(burst=burst, sustained=float(p.get("bf16_tflops_sustained", burst)),
                    hbm=float(p.get("hbm_gbs", 6650.0)), source="measured (MEASURED_PEAKS.json)")
    return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """Samples SM clock, power and throttle reasons DURING the timed region (NVML every ~5 ms in a thread;
    falls back to one nvidia-smi query if pynvml is unavailable)."""

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self._stop = threading.Event()
        self.thread = None
        self.nvml = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nvml = None
            return
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def _run(self):
        n = self.nvml
        while not self._stop.is_set():
            try:
                clk = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                pw = n.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
                rs = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle) if hasattr(
                    n, "nvmlDeviceGetCurrentClocksEventReasons") else n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                self.samples.append((clk, pw, rs))
            except Exception:
                pass
            time.sleep(0.004)

    def stop(self):
        if self.nvml is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvml unavailable"])
        self._stop.set()
        self.thread.join(timeout=2)
        if not self.samples:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        n = self.nvml
        bits = 0
        for _, _, rs in self.samples:
            bits |= rs
        names = dict(hw_slowdown=getattr(n, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                     hw_thermal_slowdown=getattr(n, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                     sw_thermal_slowdown=getattr(n, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                     sw_power_cap=getattr(n, "nvmlClocksThrottleReasonSwPowerCap", 0x4))
        reasons = sorted(k for k, v in names.items() if bits & v)
        return dict(sm_mhz=statistics.median(c for c, _, _ in self.samples), sm_max_mhz=float(self.max_sm),
                    sm_min_mhz=min(c for c, _, _ in self.samples), power_w_max=max(p for _, p, _ in self.samples),
                    samples=len(self.samples), reasons=reasons)


def synth_inputs(torch, seed, device, b=B, t=T, u=U, pin=False, view=True):
    """Synthetic batch (SURVEY 8d).  view=True: enc is generated as the encoder would deliver it, a (B,H,T) tensor, and
    handed over as its (B,T,H) permuted view (rnnt/model.py:28) -- the kernels read that layout in place."""
    g = torch.Generator().manual_seed(seed)
    enc = torch.randn(b, H, t, generator=g) if view else torch.randn(b, t, H, generator=g)
    pred = torch.randn(b, u + 1, H, generator=g)
    bound = 1.0 / (H ** 0.5)
    W = (torch.rand(V, H, generator=g) * 2 - 1) * bound
    bias = (torch.rand(V, generator=g) * 2 - 1) * bound
    targets = torch.randint(0, V - 1, (b, u), generator=g, dtype=torch.int32)
    T_len = torch.full((b,), t, dtype=torch.int32)
    U_len = torch.full((b,), u, dtype=torch.int32)
    d = dict(enc=enc, pred=pred, W=W, b=bias, targets=targets, T_len=T_len, U_len=U_len)
    d = {k: v.pin_memory() for k, v in d.items()} if pin else {k: v.to(device) for k, v in d.items()}
    if view:
        d["enc"] = d["enc"].permute(0, 2, 1)
    return d


def dump_outputs(torch, out_dir, loss, s_):
    """What one step hands its caller -- the mean loss and the gradients of enc, pred, W and b -- as float32 .npy files
    under out_dir, so that two builds can be compared output for output.  d_enc (52 MB at B=32) is kept for a fixed,
    seeded quarter of its (b, t) frames (d_enc_sample.npy, frames in ascending b * T + t order); the whole dump stays
    near 30 MB."""
    import numpy as np
    d_enc = s_["enc"].grad
    nb, nt = d_enc.shape[:2]
    frames = torch.randperm(nb * nt, generator=torch.Generator().manual_seed(0))[: nb * nt // 4].sort().values
    frames = frames.to(d_enc.device)
    arrays = dict(loss=loss.detach(), d_enc_sample=d_enc[frames // nt, frames % nt], d_pred=s_["pred"].grad,
                  dW=s_["W"].grad, db=s_["b"].grad)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.float().cpu().numpy())


# ----------------------------------------------------------------------------------------------- CPU arm
def cpu_reference_step(torch, inp):
    from oracle.ref_path import ref_loss_and_grads
    return ref_loss_and_grads(inp["enc"], inp["pred"], inp["W"], inp["b"], inp["targets"], inp["T_len"],
                              inp["U_len"], reduction="mean")


def time_cpu_reference(steps, warmup, one_thread_too=True):
    """The reference path on the host cores, BASELINE.md section 4: B=4,T=200,U=40, fp32, all threads (best of `steps`
    after `warmup`) and -- once -- a single thread.  ~10-25 s of CPU work in total."""
    import torch
    cores = os.cpu_count() or 1
    inp = synth_inputs(torch, 1234, "cpu", view=False, **{k.lower(): v for k, v in CPU_SAMPLE.items()})
    cells = CPU_SAMPLE["B"] * CPU_SAMPLE["T"] * (CPU_SAMPLE["U"] + 1)

    def best_of(n, w):
        for _ in range(w):
            cpu_reference_step(torch, inp)
        best = float("inf")
        for _ in range(n):
            t0 = time.perf_counter()
            cpu_reference_step(torch, inp)
            best = min(best, time.perf_counter() - t0)
        return best

    torch.set_num_threads(cores)
    dt = best_of(max(1, steps), warmup)
    one = None
    if one_thread_too:
        torch.set_num_threads(1)
        one = best_of(1, 0)
        torch.set_num_threads(cores)
    out = dict(value=cells / dt, unit=UNIT, cores=cores, kind="port",
               sample=f"BASELINE configs[0]: B={CPU_SAMPLE['B']},T={CPU_SAMPLE['T']},U={CPU_SAMPLE['U']},H={H},V={V} "
                      f"fp32, torch {torch.__version__} linear+tanh + torchaudio rnnt_loss fwd+bwd "
                      f"(oracle/ref_path.py = rnnt/joint.py:25-39 + rnnt/model.py:35-41), best of {max(1, steps)} after "
                      f"{warmup} warm-up, {cells} cells, {dt:.2f} s/step on {cores} threads")
    if one is not None:
        out["one_thread"] = dict(value=cells / one, unit=UNIT, cores=1, s_per_step=one)
    return out, dt


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = max(1, min(args.steps, 3))
    warmup = max(1, min(args.warmup, 1))
    base, dt = time_cpu_reference(steps, warmup)
    line = dict(metric=METRIC, value=base["value"], unit=UNIT, n_gpus=args.gpus, steps=steps, warmup=warmup,
                ms_per_step=dt * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                data="synthetic", impl="reference",
                config=dict(workload=f"joint+loss fwd+bwd on the host CPU, bounded sample: {base['sample']}"),
                cpu_baseline=base,
                e2e=dict(value=base["value"], unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------- other configs
def other_configs(torch, dev):
    """Short single-GPU runs of the remaining BASELINE.json configs (parity for these lives in tests/; this only
    reports their throughput next to the headline line)."""
    import rnnt_b200
    from rnnt_b200.functional import joint_rnnt_loss

    def timed(fn, n):
        fn(); fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    def loss_cfg(b, t, u, v, ragged, n):
        g = torch.Generator().manual_seed(77)
        enc = torch.randn(b, t, H, generator=g).to(dev).requires_grad_(True)
        pred = torch.randn(b, u + 1, H, generator=g).to(dev).requires_grad_(True)
        bound = 1.0 / (H ** 0.5)
        W = ((torch.rand(v, H, generator=g) * 2 - 1) * bound).to(dev).requires_grad_(True)
        bias = ((torch.rand(v, generator=g) * 2 - 1) * bound).to(dev).requires_grad_(True)
        tg = torch.randint(0, v - 1, (b, u), generator=g, dtype=torch.int32).to(dev)
        if ragged:
            tl = torch.randint(t // 2, t + 1, (b,), generator=g, dtype=torch.int32); tl[0] = t
            ul = torch.randint(u // 2, u + 1, (b,), generator=g, dtype=torch.int32); ul[-1] = u
        else:
            tl = torch.full((b,), t, dtype=torch.int32); ul = torch.full((b,), u, dtype=torch.int32)
        cells = int((tl.long() * (ul.long() + 1)).sum())
        tl, ul = tl.to(dev), ul.to(dev)

        def fn():
            for x in (enc, pred, W, bias):
                x.grad = None
            joint_rnnt_loss(enc, pred, W, bias, tg, tl, ul, validate=False).backward()
        torch.cuda.reset_peak_memory_stats(dev)
        ms = timed(fn, n)
        return dict(ms_per_step=ms, valid_cells=cells, value=cells / (ms * 1e-3), unit=UNIT,
                    peak_mem_gib=torch.cuda.max_memory_allocated(dev) / 2 ** 30)

    out = {}
    # context only: the ops the reference's call path launches on a GPU (cuBLAS fp32 linear + tanh + torchaudio's
    # CUDA rnnt_loss, materialised logits), timed on this GPU at a batch that fits
    try:
        import torchaudio
        ri = synth_inputs(torch, 4242, dev, b=8)
        for k in ("enc", "pred", "W", "b"):
            ri[k].requires_grad_(True)

        def ref_gpu_step():
            for k in ("enc", "pred", "W", "b"):
                ri[k].grad = None
            hid = torch.tanh(ri["enc"].unsqueeze(2) + ri["pred"].unsqueeze(1))
            logits = torch.nn.functional.linear(hid, ri["W"], ri["b"])
            torchaudio.functional.rnnt_loss(logits, ri["targets"], ri["T_len"], ri["U_len"], blank=-1, clamp=-1,
                                            reduction="mean").backward()
        ms = timed(ref_gpu_step, 3)
        out["reference_ops_on_this_gpu_B8_T400_U100_V1024"] = dict(
            ms_per_step=ms, value=8 * T * (U + 1) / (ms * 1e-3), unit=UNIT,
            note="torch fp32 linear + tanh + torchaudio CUDA rnnt_loss fwd+bwd; context, not the contract's reference arm")
        del ri
        torch.cuda.empty_cache()
    except Exception as exc:
        out["reference_ops_on_this_gpu_B8_T400_U100_V1024"] = dict(error=repr(exc))
    out["cpu_reference_shape_B4_T200_U40_V1024"] = loss_cfg(4, 200, 40, 1024, False, 20)
    out["ragged_B32_T400_U100_V1024"] = loss_cfg(32, 400, 100, 1024, True, 5)
    out["stress_B8_T1500_U300_V4096_ragged"] = loss_cfg(8, 1500, 300, 4096, True, 2)
    # batched greedy decode (BASELINE configs[4]): B=64, T=400, ConvPredictor at default init, max_length 200 -- the
    # round-1 workload (blank bias +1.0: every utterance emits until max_length, so EVERY step runs the predictor phases)
    import rnnt_b200.functional as RF
    torch.manual_seed(0)
    E = 512
    joint = rnnt_b200.JointNetwork(-1, -1, H, V)
    with torch.no_grad():
        joint.joint_ln.bias[V - 1] += 1.0
    model = rnnt_b200.RNNTModel(rnnt_b200.ConvPredictor(V, H, E, 0.3), torch.nn.Identity(), joint).eval()
    feats_cpu = torch.randn(64, 400, H)
    lens = torch.randint(200, 401, (64,)); lens[0] = 400
    # the reference's own loop (rnnt/model.py:90-128 restated in oracle/ref_path.py) on the host cores, 4 utterances
    from oracle.ref_path import ref_greedy_decode
    sd = {k: v.detach() for k, v in model.predictor.state_dict().items()}
    n_ref = 4
    torch.set_num_threads(os.cpu_count() or 1)
    t0 = time.perf_counter()
    ref_toks = [ref_greedy_decode(feats_cpu[i:i + 1, : int(lens[i])], joint.joint_ln.weight.detach(),
                                  joint.joint_ln.bias.detach(), sd, V - 1, 200) for i in range(n_ref)]
    cpu_s = time.perf_counter() - t0
    cpu_frames = int(lens[:n_ref].sum())
    model = model.to(dev)
    feats = feats_cpu.to(dev)
    model.greedy_decode_features(feats, lens, max_length=200)
    torch.cuda.synchronize()
    best = float("inf")
    for _ in range(3):
        t0 = time.perf_counter()
        toks = model.greedy_decode_features(feats, lens, max_length=200)
        torch.cuda.synchronize()
        best = min(best, time.perf_counter() - t0)
    cyc = RF._last_decode_phase_cycles.tolist()
    frames, ntok = int(lens.sum()), sum(len(x) for x in toks)
    steps = int(cyc[6])                                               # joint steps the kernel took (its own counter)
    w_bytes = 4 * (V * H + E * 5 * E + H * E)                         # fp32 weights a step multiplies with (shared memory)
    out["greedy_decode_B64_T400"] = dict(
        ms_total=best * 1e3, frames=frames, frames_per_s=frames / best, tokens=ntok, steps=steps,
        us_per_step=best * 1e6 / steps, weight_bytes_per_step=w_bytes, l2_gbs=w_bytes * steps / best / 1e9,
        bound="latency: one cooperative kernel, 5 grid barriers per emitting step (1.2 us each + waiting for the slowest "
              "CTA of the phase); the fp32 weights (11.5 MB: joint, conv2, linear) are resident in shared memory (82 KB "
              "per SM), conv1 is a per-symbol table built at kernel start, a step only moves activations through L2, so "
              "neither HBM nor the tensor pipe is the limit",
        phase_cycles=dict(zip(["P1", "P2", "P3", "conv1_table_build", "P5", "P6", "steps", "grid_barriers"], cyc)),
        tokens_match_cpu_reference=[toks[i] == ref_toks[i] for i in range(n_ref)],
        cpu_reference=dict(frames_per_s=cpu_frames / cpu_s, s_total=cpu_s, utterances=n_ref, frames=cpu_frames,
                           cores=os.cpu_count(), kind="port",
                           note="rnnt/model.py:90-128 restated (oracle/ref_path.py), one utterance at a time"),
        note="whole batched loop in one persistent kernel, wall clock incl. result read-back, best of 3")
    return out


# ----------------------------------------------------------------------------------------------- GPU arm
KERNEL_FAMILIES = ["prep", "joint_gemm_fwd", "lattice", "joint_gemm_bwd", "dh_gemm", "dw_gemm", "db", "other"]
GEMM_FAMILIES = ("joint_gemm_fwd", "joint_gemm_bwd", "dh_gemm", "dw_gemm")


def kernel_table(fam_ms, fam_n, nsteps, ms_step, cells_rank, bwd_frac, peak_tflops, hbm_peak):
    """Per kernel family: ms per step, share of the step, achieved TFLOP/s on the FLOPs it executed (the backward GEMMs
    only run over half-tiles with non-zero gradients) and that as a fraction of `peak_tflops`."""
    kern = {}
    gemm_flops = cells_rank * FLOP_PER_CELL_GEMM
    for i, nm in enumerate(KERNEL_FAMILIES):
        if fam_n[i] == 0:
            continue
        per_step_ms = fam_ms[i] / nsteps
        k = dict(ms_per_step=per_step_ms, launches_per_step=fam_n[i] / nsteps, share=per_step_ms / ms_step)
        if nm in GEMM_FAMILIES:
            frac = 1.0 if nm == "joint_gemm_fwd" else bwd_frac
            k["flops_per_step"] = gemm_flops * frac
            k["tflops"] = gemm_flops * frac / (per_step_ms * 1e-3) / 1e12
            k["frac_of_peak"] = k["tflops"] / peak_tflops
        if nm == "lattice":
            # algorithmic bytes: each direction reads lp (8 B/cell) and writes alpha or beta (4 B/cell).  The kernel is
            # bound by the (T+U)-step dependency chain of the wavefront (one CTA per utterance and direction), not by HBM.
            k["gbs"] = cells_rank * 24 / (per_step_ms * 1e-3) / 1e9
            k["hbm_frac"] = k["gbs"] / hbm_peak
            k["ns_per_antidiagonal"] = per_step_ms * 1e6 / (T + U)
            k["bound"] = "latency: T+U dependent anti-diagonal steps, 2*B CTAs"
        kern[nm] = k
    return kern


def run_gpu_arm(args):
    import torch
    import torch.distributed as dist
    from rnnt_b200 import _lib
    import rnnt_b200.functional as RF
    from rnnt_b200.functional import joint_rnnt_loss
    from rnnt_b200.parallel import WeightGradBucket
    os.environ.setdefault("NCCL_DEBUG", "WARN")     # keep NCCL's banner off stdout: rank 0 prints ONE JSON line

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L = _lib.lib()

    # workload: N=1 -> configs[1] (B=32); N>1 -> configs[2] (global 256 sharded by utterance) unless --global-batch 0
    strong = world > 1 and args.global_batch > 0
    if strong and args.global_batch % world:
        raise SystemExit(f"--global-batch {args.global_batch} must divide by the number of GPUs ({world})")
    Bg = args.global_batch // world if strong else B
    cells_rank = Bg * T * (U + 1)

    def make_sets(b, n_sets=3):   # rotating input sets: >= 3 x 70 MB > 126 MB L2, so inputs are L2-cold every step
        sets = [synth_inputs(torch, 1234 + rank * 16 + i, dev, b=b, view=not args.dense_encoder) for i in range(n_sets)]
        for s_ in sets:
            for k in ("enc", "pred", "W", "b"):
                s_[k].requires_grad_(True)
        return sets

    sets = make_sets(Bg)
    bucket = None
    if world > 1:      # dW / db are written straight into the flat all-reduce bucket; predictor grads ride as a stub
        bucket = WeightGradBucket(V, H, PRED_GRAD_ELEMS, dev, average=True)
        bucket.time_collectives = True
        RF.set_weight_grad_sink(bucket)

    def step(s_, all_tiles=False):
        for k in ("enc", "pred", "W", "b"):
            s_[k].grad = None
        loss = joint_rnnt_loss(s_["enc"], s_["pred"], s_["W"], s_["b"], s_["targets"], s_["T_len"], s_["U_len"],
                               blank=-1, clamp=-1, reduction="mean", validate=False,
                               skip_zero_tiles=not (all_tiles or args.all_tiles))
        loss.backward()          # with a bucket: the all-reduce of dW/db is already in flight under the dh GEMM
        if bucket is not None:
            bucket.finish()      # predictor stub slice + averaging; the compute stream waits for the result
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_region(nsteps, use_sets, profile, sample_clocks, **kw):
        sampler = ClockSampler(local_rank)
        if sample_clocks and rank == 0:
            sampler.start()
        if bucket is not None:
            bucket.reset_timing()
        if profile:
            L.rnnt_b200_profile_begin()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        last = None
        for i in range(nsteps):
            last = step(use_sets[i % len(use_sets)], **kw)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        fam_ms, fam_n = (C.c_float * 8)(), (C.c_int64 * 8)()
        if profile:
            _lib.check(L.rnnt_b200_profile_end(fam_ms, fam_n), "profile_end")
        clocks = sampler.stop() if (sample_clocks and rank == 0) else None
        nccl_ms = bucket.collective_ms() / nsteps if bucket is not None else 0.0
        exposed_ms = bucket.exposed_ms() / nsteps if bucket is not None else 0.0
        return dict(ms=ms, fam_ms=list(fam_ms), fam_n=list(fam_n), clocks=clocks, last=last, nccl_ms=nccl_ms,
                    exposed_ms=exposed_ms)

    for i in range(args.warmup):
        step(sets[i % len(sets)])
    barrier()

    # ---- headline timed region: K steps, CUDA events on the launch stream, clocks sampled, per-kernel events on
    head = timed_region(args.steps, sets, not args.no_kernel_profile, True)
    ms_total = head["ms"]
    loss_val = float(head["last"].detach())
    if args.dump_outputs and rank == 0:     # before the secondary loops below overwrite the gradients of these sets
        dump_outputs(torch, args.dump_outputs, head["last"], sets[(args.steps - 1) % len(sets)])

    # ---- secondary numbers (single GPU only): every tile in the backward; a >= 3 s sustained loop under the power cap
    dense_ms, sustained = None, None
    if world == 1 and not args.all_tiles:
        for i in range(2):
            step(sets[i % len(sets)], all_tiles=True)
        dense_ms = timed_region(max(2, args.steps // 2), sets, False, False, all_tiles=True)["ms"] / max(2, args.steps // 2)
    if world == 1 and args.sustain_s > 0:
        n_sus = max(args.steps, int(args.sustain_s * 1e3 / (ms_total / args.steps)) + 1)
        sus = timed_region(n_sus, sets, not args.no_kernel_profile, True)
        sustained = dict(steps=n_sus, ms_per_step=sus["ms"] / n_sus, seconds=sus["ms"] * 1e-3, clocks=sus["clocks"],
                         fam_ms=sus["fam_ms"], fam_n=sus["fam_n"])
    RF.COLLECT_BACKWARD_STATS = True
    step(sets[0])
    torch.cuda.synchronize()
    active_tiles, total_tiles = RF.last_backward_stats()
    RF.COLLECT_BACKWARD_STATS = False
    bwd_frac = active_tiles / max(1, total_tiles)

    # ---- round-1 workload for continuity (N>1 only): weak scaling, B=32 per GPU
    weak_ms = None
    if strong:
        del sets
        torch.cuda.empty_cache()
        wsets = make_sets(B)
        for i in range(3):
            step(wsets[i % 3])
        weak_ms = timed_region(max(5, args.steps // 2), wsets, False, False)["ms"] / max(5, args.steps // 2)
        del wsets
        torch.cuda.empty_cache()

    # ---- e2e: same step through the public API from pinned HOST buffers, result read back to host.
    # Every step copies that step's inputs host->device (all 7 tensors) and reads its loss back; the copy of
    # step i+1 runs on a side stream into the other device buffer while step i computes (double buffering).
    host = synth_inputs(torch, 4321 + rank, dev, b=Bg, pin=True, view=not args.dense_encoder)
    devbufs = []
    for _ in range(2):
        d = {k: torch.empty_like(v, device=dev) for k, v in host.items()}      # keeps the (B,H,T)-view strides of enc
        for k in ("enc", "pred", "W", "b"):
            d[k].requires_grad_(True)
        devbufs.append(d)
    h2d = sum(v.numel() * v.element_size() for v in host.values())
    host_loss = torch.empty((), dtype=torch.float32).pin_memory()
    copy_stream = torch.cuda.Stream(device=dev)
    copied = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]

    def enqueue_copy(i):
        buf = devbufs[i & 1]
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[i & 1])          # the step that last used this buffer has finished
            with torch.no_grad():
                for k, v in host.items():
                    buf[k].copy_(v, non_blocking=True)
            copied[i & 1].record(copy_stream)

    def e2e_loop(n):
        for j in (0, 1):
            consumed[j].record(torch.cuda.current_stream())
        enqueue_copy(0)
        val = 0.0
        for i in range(n):
            if i + 1 < n:
                enqueue_copy(i + 1)
            torch.cuda.current_stream().wait_event(copied[i & 1])
            loss = step(devbufs[i & 1])
            consumed[i & 1].record(torch.cuda.current_stream())
            host_loss.copy_(loss.detach(), non_blocking=True)
            torch.cuda.current_stream().synchronize()        # the step's result is on the host before the next step
            val = float(host_loss)
        return val

    e2e_loop(min(2, args.warmup))
    barrier()
    t0 = time.perf_counter()
    e2e_loop(args.steps)
    barrier()
    e2e_s = time.perf_counter() - t0

    # ---- max over ranks
    times = torch.tensor([ms_total, e2e_s * 1e3, dense_ms or 0.0, weak_ms or 0.0, head["nccl_ms"], head["exposed_ms"]],
                         dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    ms_total, e2e_ms, dense_ms, weak_ms, nccl_ms, exposed_ms = (float(x) for x in times)

    if rank == 0:
        peaks = load_peaks()
        cells_step = cells_rank * world
        ms_step = ms_total / args.steps
        value = cells_step / (ms_step * 1e-3)
        # regime of the headline timed region: a short burst runs at boost clocks, seconds-long loops at the power cap
        regime = "sustained" if ms_total >= 2000.0 else "burst"
        head_peak = peaks[regime]
        kern = kernel_table(head["fam_ms"], head["fam_n"], args.steps, ms_step, cells_rank, bwd_frac, head_peak,
                            peaks["hbm"])
        gemms = {k: v for k, v in kern.items() if "tflops" in v}
        if not gemms:   # --no-kernel-profile: no per-kernel events were recorded
            gemms = {"whole_step": dict(ms_per_step=ms_step, launches_per_step=1.0,
                                        tflops=(1 + 3 * bwd_frac) * cells_rank * FLOP_PER_CELL_GEMM / (ms_step * 1e-3) / 1e12)}
        dom = max(gemms, key=lambda k: gemms[k]["ms_per_step"])
        launches_dom = gemms[dom]["launches_per_step"]
        achieved = gemms[dom]["tflops"]
        traffic = None
        import glob
        tfiles = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")))
        tpath = tfiles[-1] if tfiles else ""
        if tpath:     # DRAM bytes per launch of that kernel from the latest committed ncu --set full capture
            with open(tpath) as f:
                traffic = json.load(f).get(dom, {}).get("dram_bytes_per_launch")
        exec_flops_rank = (1 + 3 * bwd_frac) * cells_rank * FLOP_PER_CELL_GEMM     # F over all tiles; G, dh, dW over active ones
        per_gpu_cells_s = value / world
        roofline = dict(
            bound="tensor", kernel=dom, achieved=achieved, peak=head_peak, unit="TFLOP/s", frac=achieved / head_peak,
            regime=f"{regime}: the headline timed region lasted {ms_total * 1e-3:.2f} s, so the denominator is the "
                   f"{'burst (best-of-10)' if regime == 'burst' else 'sustained (4 s loop)'} cuBLAS bf16 figure",
            traffic=traffic, peak_source=peaks["source"],
            flops_per_launch=gemms[dom].get("flops_per_step", cells_rank * FLOP_PER_CELL_GEMM) / launches_dom,
            avg_launch_ms=gemms[dom]["ms_per_step"] / launches_dom,
            whole_step_frac_executed=exec_flops_rank / (ms_step * 1e-3) / 1e12 / head_peak,
            whole_step_frac_crediting_skipped_tiles=per_gpu_cells_s * 3 * FLOP_PER_CELL_GEMM / (head_peak * 1e12),
            note="whole_step_frac_executed counts the FLOPs the GEMM kernels really ran (2HV per cell in the forward, "
                 "6HV per cell of an ACTIVE half-tile in the backward incl. the logit recompute); "
                 "..._crediting_skipped_tiles credits the algorithmic 6HV on every cell, also those the backward "
                 "skipped, so it is a throughput figure, not a utilisation",
            kernels=kern)
        if sustained is not None:
            sk = kernel_table(sustained["fam_ms"], sustained["fam_n"], sustained["steps"], sustained["ms_per_step"],
                              cells_rank, bwd_frac, peaks["sustained"], peaks["hbm"])
            sg = {k: v for k, v in sk.items() if "tflops" in v}
            roofline["sustained"] = dict(
                seconds=sustained["seconds"], steps=sustained["steps"], ms_per_step=sustained["ms_per_step"],
                value=cells_rank / (sustained["ms_per_step"] * 1e-3), unit=UNIT, peak=peaks["sustained"],
                kernel=dom, achieved=sg[dom]["tflops"] if dom in sg else None,
                frac=sg[dom]["tflops"] / peaks["sustained"] if dom in sg else None,
                whole_step_frac_executed=exec_flops_rank / (sustained["ms_per_step"] * 1e-3) / 1e12 / peaks["sustained"],
                clocks=sustained["clocks"], kernels=sk)
        cpu_base, _ = time_cpu_reference(3, 1) if world == 1 and not args.no_cpu_baseline else (None, None)
        extra = None
        if world == 1 and not args.no_extra:
            try:
                extra = other_configs(torch, dev)
            except Exception as exc:      # the headline line must not depend on the side runs
                extra = dict(error=repr(exc))
        if strong:
            workload = (f"BASELINE configs[2]: global batch {args.global_batch} sharded by utterance, "
                        f"{Bg} per GPU in one launch (T={T},U={U},H={H},V={V}), joint+loss fused fwd+bwd")
        else:
            workload = (f"BASELINE configs[1]: joint+loss fused fwd+bwd, per-GPU B={B},T={T},U={U},H={H},V={V}; "
                        f"global batch {B * world}")
        line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=ms_step, higher_is_better=True, scaling="strong" if strong else "weak",
                    vs_baseline=None, dtype="fp16", data="synthetic",
                    config=dict(workload=workload, global_batch=Bg * world, per_gpu_batch=Bg,
                                parallelism=(f"dp{world} by utterance; dW/db written into one flat bucket, NCCL "
                                             f"all-reduce of {V * H + V} joint + {PRED_GRAD_ELEMS} predictor(stub) fp32 "
                                             "grads, the joint part overlapped with the dh GEMM") if world > 1 else "single GPU",
                                encoder_layout=("dense (B,T,H) tensor (--dense-encoder)" if args.dense_encoder else
                                                "(B,T,H) view of a (B,H,T) tensor (rnnt/model.py:28), read in place"),
                                l2=f"3 rotating input sets ({3 * 70 * Bg // 32} MB > 126 MB L2); every step also streams the "
                                   "fp16 activation residual and the gradient ring through HBM",
                                operands="fp16 x fp16 -> fp32 (TMEM), fp32 elsewhere",
                                backward_tiles=dict(active=active_tiles, total=total_tiles, fraction=bwd_frac,
                                                    note="half-tiles (16 t x 4 u lattice blocks) whose fp16 logit-"
                                                         "gradients are all zero (occupancy < 2^-25) are skipped; "
                                                         "--all-tiles disables"),
                                loss=loss_val),
                    clocks=head["clocks"],
                    e2e=dict(value=cells_step / (e2e_ms * 1e-3 / args.steps), unit=UNIT,
                             h2d_bytes_per_step=h2d, d2h_bytes_per_step=4, ms_per_step=e2e_ms / args.steps),
                    gpu_launches=int(sum(head["fam_n"])),
                    all_tiles=(dict(ms_per_step=dense_ms, value=cells_step / (dense_ms * 1e-3), unit=UNIT,
                                    frac_credited=cells_rank * 3 * FLOP_PER_CELL_GEMM / (dense_ms * 1e-3) / 1e12 / head_peak,
                                    frac_executed=cells_rank * 4 * FLOP_PER_CELL_GEMM / (dense_ms * 1e-3) / 1e12 / head_peak,
                                    note="same step, backward over every half-tile of the lattice (zero-gradient ones "
                                         "not skipped): the data-independent number; credited = 6HV per cell, executed "
                                         "= 8HV per cell (the backward recomputes the logits)")
                               if dense_ms else None),
                    roofline=roofline)
        if world > 1:
            line["nccl"] = dict(exposed_ms_per_step=exposed_ms, in_flight_ms_per_step=nccl_ms,
                                bytes_per_step=4 * (V * H + V + PRED_GRAD_ELEMS),
                                note="exposed = time the compute stream stalls for the collectives at the end of the "
                                     "step (CUDA events, max over ranks); in_flight = enqueue-to-completion of the "
                                     "all-reduces on the side stream (the joint bucket's is gated by the dW-done event "
                                     "and shares the SMs with the dh GEMM, so it includes waiting for SM resources)")
        if weak_ms:
            line["weak_b32_per_gpu"] = dict(ms_per_step=weak_ms, value=B * T * (U + 1) * world / (weak_ms * 1e-3),
                                            unit=UNIT, global_batch=B * world,
                                            note="round-1 workload for continuity: B=32 per GPU, weak scaling")
        if cpu_base is not None:
            line["cpu_baseline"] = cpu_base
        if extra is not None:
            line["other_configs"] = extra
        print(json.dumps(line), flush=True)
    RF.set_weight_grad_sink(None)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kernel-profile", action="store_true", help="skip the per-kernel CUDA events")
    ap.add_argument("--no-extra", action="store_true", help="skip the short runs of the other BASELINE.json configs")
    ap.add_argument("--global-batch", type=int, default=GLOBAL_BATCH,
                    help="N>1: global batch sharded over the GPUs (BASELINE configs[2]); 0 = weak scaling, B=32 per GPU")
    ap.add_argument("--sustain-s", type=float, default=3.0,
                    help="N=1: length of the extra sustained (power-capped) loop in seconds; 0 disables")
    ap.add_argument("--dense-encoder", action="store_true",
                    help="feed a dense (B,T,H) encoder tensor instead of the (B,H,T) view the reference model produces")
    ap.add_argument("--all-tiles", action="store_true",
                    help="backward processes every half-tile of the lattice (also those whose fp16 gradients are all zero)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss and gradients of the last timed step to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
