#!/usr/bin/env python
"""bench.py -- headline benchmark: HiFi-GAN v1 (22.05 kHz) generator inference,
BASELINE.json configs[1]: batch 16 x 80 x 400 synthetic mels -> 16 x 1 x 102400 samples.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one generator forward over one batch.  Multi-GPU (torchrun, one rank per
GPU): independent utterance batches per rank, no data-path collective ("weak" scaling);
time = max over ranks (device events), value = total samples / that time.

Output: ONE JSON line on rank 0 with the extra objects `roofline`, `cpu_baseline`, `e2e`,
`clocks`, `gpu_launches`.  `--dump-outputs DIR` also writes the audio the last timed step
returned as DIR/audio.npy (float32, 16 x 1 x 102400; DIR/audio_rank<r>.npy per rank when
N > 1).  Weights and mels are seeded, so two builds run with the same arguments can be
compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

FS = 22050
CFG = dict(in_channels=80, out_channels=1, channels=512, kernel_size=7, upsample_scales=[8, 8, 2, 2],
           upsample_kernel_sizes=[16, 16, 4, 4], resblock_kernel_sizes=[3, 7, 11],
           resblock_dilations=[[1, 3, 5], [1, 3, 5], [1, 3, 5]], use_additional_convs=True, bias=True,
           nonlinear_activation="LeakyReLU", nonlinear_activation_params={"negative_slope": 0.1})
BATCH, FRAMES, HOP = 16, 400, 256
METRIC = "audio_samples_per_sec"
UNIT = "samples/s"
WORKLOAD = "HiFi-GAN v1 generator inference (ljspeech hifigan.v1.yaml), 16x80x400 mels -> 16x1x102400 samples, fp32 weights, weight-norm folded"


def synth_weights(seed=1234):
    """Random-init weights of the HiFi-GAN v1 architecture (no checkpoints offline): synthetic
    state dict in the reference layout, folded (remove_weight_norm) like decode.py:147."""
    from parallelwavegan_b200 import synth_weights as synth  # seeded random-init weights (no checkpoints offline)
    from parallelwavegan_b200 import models

    m = models.HiFiGANGenerator(**CFG)
    spec = [(k, tuple(v.shape)) for k, v in m.state_dict().items()]
    sd = synth.synth_state_dict(spec, seed, 1.15)
    m.load_state_dict(sd)
    m.remove_weight_norm()
    return m.eval(), sd


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                smax = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


def shared_config(world):
    """`config` of BOTH arms (ours and --impl reference): the workload only, nothing implementation specific."""
    return {"workload": WORKLOAD, "per_gpu_batch": BATCH, "frames": FRAMES, "mel_channels": 80, "hop": HOP, "fs": FS,
            "weights": "random-init HiFi-GAN v1 (seeded synthetic state dict), weight norm folded",
            "parallelism": f"utterance-sharded x{world}"}


def cpu_reference_forward(weights, c):
    """The reference's CPU implementation of the path, restated (oracle port): same ATen CPU ops."""
    from oracle import ref_ops

    with torch.no_grad():
        return ref_ops.hifigan_generator(weights, c, dict(CFG, negative_slope=0.1))


def tune_cpu_threads(weights):
    """The oneDNN/ATen CPU path does not scale to every core of a big host (128-core box: 13-19 k
    samples/s with 128 threads).  Give the reference its best thread count: probe a few."""
    cores = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, cores) if c <= cores})
    probe = torch.randn(1, 80, 64)
    best, best_t = cores, None
    for c in cands:
        torch.set_num_threads(c)
        cpu_reference_forward(weights, probe)
        t0 = time.perf_counter()
        cpu_reference_forward(weights, probe)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best, cores


def cpu_decode_batch(weights, c):
    """ONE protocol for every CPU leg: the batch is decoded utterance by utterance, exactly like the
    reference's own decode loop (bin/decode.py:214-243 calls model.inference once per utterance)."""
    n = 0
    for i in range(c.shape[0]):
        n += cpu_reference_forward(weights, c[i : i + 1]).numel()
    return n


def time_cpu(weights, batch, frames, reps):
    c = torch.randn(batch, 80, frames)
    cpu_reference_forward(weights, torch.randn(1, 80, 16))  # warm-up (thread pool, oneDNN primitives)
    best = None
    for _ in range(reps):
        t0 = time.perf_counter()
        n = cpu_decode_batch(weights, c)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return n / best, best


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU path (oracle port; /root/reference does not exist
    on the GPU box) on all host cores, one bounded sample per step."""
    if rank != 0:
        return
    from oracle.ref_ops import fold_weight_norm

    _, sd = synth_weights()
    w = fold_weight_norm(sd)
    cores, host_cores = tune_cpu_threads(w)
    # the full workload every step: all 16 utterances of the 16x80x400 batch (decoded one by one like
    # bin/decode.py does); warm-up steps run on short mels (they only warm the thread pool / oneDNN)
    c = torch.randn(BATCH, 80, FRAMES, generator=torch.Generator().manual_seed(100))
    for _ in range(max(args.warmup, 1)):
        cpu_reference_forward(w, c[:1, :, :64])
    t0 = time.perf_counter()
    n = 0
    for _ in range(args.steps):
        n += cpu_decode_batch(w, c)
    dt = time.perf_counter() - t0
    val = n / dt
    sample = (f"the full {BATCH}x80x{FRAMES} batch every step, utterance by utterance (bin/decode.py:214-243), {args.steps} steps, "
              f"torch CPU fp32 (oracle port), {cores} threads (best of a probe over 8..{host_cores} on a {host_cores}-core host)")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": shared_config(world),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "rtf": FS / val,
    }))


def measure_train_step(dev, rank, local_rank, world, dist, steps=3, warmup=2):
    """Secondary metric (BASELINE.json "train steps/sec"): HiFi-GAN v1 G + MSD/MPD full train step
    (C5: per-GPU batch 16 x 8192 samples; mel + adversarial + feature-matching losses, Adam), forward and
    backward on libpwgb kernels, DDP gradient all-reduce over NCCL when world > 1."""
    from parallelwavegan_b200 import losses, models
    from parallelwavegan_b200 import synth_weights as synth
    from parallelwavegan_b200.train_step import GanTrainStep

    g = models.HiFiGANGenerator(**CFG)
    g.load_state_dict(synth.synth_state_dict([(k, tuple(v.shape)) for k, v in g.state_dict().items()], 1234, 1.15))
    d = models.HiFiGANMultiScaleMultiPeriodDiscriminator()
    d.load_state_dict(synth.synth_state_dict([(k, tuple(v.shape)) for k, v in d.state_dict().items()], 4321, 1.4))
    g, d = g.to(dev).train(), d.to(dev).train()
    if world > 1:
        g = torch.nn.parallel.DistributedDataParallel(g, device_ids=[local_rank])
        d = torch.nn.parallel.DistributedDataParallel(d, device_ids=[local_rank])
    crit = {"mel": losses.MelSpectrogramLoss(fs=22050, fft_size=1024, hop_size=256, win_length=None, window="hann", num_mels=80,
                                             fmin=0, fmax=11025, log_base=None).to(dev),
            "gen_adv": losses.GeneratorAdversarialLoss(), "dis_adv": losses.DiscriminatorAdversarialLoss(),
            "feat_match": losses.FeatureMatchLoss()}
    from parallelwavegan_b200.optimizers import FusedAdam

    step = GanTrainStep(g, d, crit, FusedAdam(g.parameters(), lr=2e-4, betas=(0.5, 0.9)),
                        FusedAdam(d.parameters(), lr=2e-4, betas=(0.5, 0.9)), lambda_aux=45.0, lambda_adv=1.0, lambda_feat_match=2.0,
                        steps=1)
    gen = torch.Generator().manual_seed(1000 + rank)
    c = torch.randn(16, 80, 32, generator=gen).to(dev)
    y = (torch.rand(16, 1, 8192, generator=gen) - 0.5).to(dev)
    for _ in range(warmup):
        st = step(c, y)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        st = step(c, y)
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    return {"metric": "train_steps_per_sec", "value": 1e3 / ms, "ms_per_step": ms, "global_batch": 16 * world,
            "workload": "HiFi-GAN v1 G + MSD/MPD train step, per-GPU batch 16 x 8192 samples (hifigan.v1.yaml losses, Adam)",
            "parallelism": f"DDP x{world} (NCCL gradient all-reduce)" if world > 1 else "single GPU",
            "losses": {k: float(v) for k, v in st.items()}}


def measure_pwg_train_step(dev, rank, local_rank, world, dist, steps=3, warmup=2, batch=64):
    """BASELINE.json configs[2]: Parallel WaveGAN v1 G + D train step (30-layer residual stack,
    MultiResolutionSTFTLoss + adversarial loss, RAdam), per-GPU batch 64 x 25600 samples, DDP when world > 1."""
    from parallelwavegan_b200 import losses, models
    from parallelwavegan_b200 import synth_weights as synth

    g = models.ParallelWaveGANGenerator()
    g.load_state_dict(synth.synth_state_dict([(k, tuple(v.shape)) for k, v in g.state_dict().items()], 31, 1.0))
    d = models.ParallelWaveGANDiscriminator()
    d.load_state_dict(synth.synth_state_dict([(k, tuple(v.shape)) for k, v in d.state_dict().items()], 64, 1.4))
    g, d = g.to(dev).train(), d.to(dev).train()
    if world > 1:  # the last layer's residual 1x1 has no influence on the output (parallel_wavegan.py:161-166)
        g = torch.nn.parallel.DistributedDataParallel(g, device_ids=[local_rank], find_unused_parameters=True)
        d = torch.nn.parallel.DistributedDataParallel(d, device_ids=[local_rank])
    from parallelwavegan_b200.optimizers import RAdam
    from parallelwavegan_b200.train_step import GanTrainStep

    crit = {"stft": losses.MultiResolutionSTFTLoss().to(dev), "gen_adv": losses.GeneratorAdversarialLoss(),
            "dis_adv": losses.DiscriminatorAdversarialLoss()}
    # parallel_wavegan.v1.yaml:67-108: lambda_adv 4.0, RAdam lr 1e-4 / 5e-5 eps 1e-6, grad clip 10 / 1
    tstep = GanTrainStep(g, d, crit, RAdam(g.parameters(), lr=1e-4, eps=1e-6), RAdam(d.parameters(), lr=5e-5, eps=1e-6),
                         lambda_aux=1.0, lambda_adv=4.0, grad_norm_g=10.0, grad_norm_d=1.0, steps=1)
    T = 25600
    gen = torch.Generator().manual_seed(2000 + rank)
    c = torch.randn(batch, 80, T // 256 + 4, generator=gen).to(dev)
    y = (torch.rand(batch, 1, T, generator=gen) - 0.5).to(dev)

    def step():
        z = torch.randn(batch, 1, T, device=dev)
        st = tstep((z, c), y)
        return st["generator_loss"], st["discriminator_loss"]

    for _ in range(warmup):
        st = step()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        st = step()
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    return {"metric": "train_steps_per_sec", "value": 1e3 / ms, "ms_per_step": ms, "global_batch": batch * world,
            "workload": f"ParallelWaveGAN v1 G + D train step, per-GPU batch {batch} x {T} samples (parallel_wavegan.v1.yaml losses, RAdam)",
            "parallelism": f"DDP x{world} (NCCL gradient all-reduce)" if world > 1 else "single GPU",
            "losses": {"generator_loss": float(st[0]), "discriminator_loss": float(st[1])}}


def measure_batch1(model, dev, flush, steps=20):
    """north_star RTF target: HiFi-GAN v1 at batch 1 (1 x 80 x 400 mels = 4.64 s of audio), eager launches and
    CUDA-graph replay (decode driver), L2 flushed between steps, device events."""
    from parallelwavegan_b200 import decode

    c1 = torch.randn(1, 80, FRAMES, generator=torch.Generator().manual_seed(7)).to(dev)
    out = {"workload": f"1x80x{FRAMES} mels -> {FRAMES * HOP} samples ({FRAMES * HOP / FS:.2f} s of audio)"}
    with torch.no_grad():
        runner = decode.GraphedGenerator(model)
        for name, fn in (("eager", model), ("cuda_graph", runner)):
            for _ in range(3):
                fn(c1)
            torch.cuda.synchronize()
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
            for e0, e1 in evs:
                flush.zero_()
                e0.record()
                fn(c1)
                e1.record()
            torch.cuda.synchronize()
            ms = statistics.median(e0.elapsed_time(e1) for e0, e1 in evs)
            out[name] = {"ms": ms, "rtf": ms * 1e-3 / (FRAMES * HOP / FS), "x_realtime": (FRAMES * HOP / FS) / (ms * 1e-3)}
    return out


def _time_cuda(fn, steps, warmup, flush):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for e0, e1 in evs:
        flush.zero_()
        e0.record()
        fn()
        e1.record()
    torch.cuda.synchronize()
    return sum(e0.elapsed_time(e1) for e0, e1 in evs) / steps


def measure_torch_eager_gpu(dev, sd, mel_dev, flush):
    """The honest GPU comparison (BASELINE.md section 3 item 5): the reference's algorithm as plain PyTorch eager ops
    (cuDNN / cuBLAS / cuFFT; the oracle port run on CUDA tensors, weight norm folded) on the SAME B200, for the C2
    forward (TF32 off = fp32 parity class, and on) and the C5 train step.  A baseline, measured in the same run."""
    import torch.nn.functional as F

    from oracle import ref_ops
    from oracle.ref_ops import fold_spectral_norm_eval, fold_weight_norm
    from parallelwavegan_b200 import models
    from parallelwavegan_b200 import synth_weights as synth

    out = {"what": "reference algorithm as PyTorch eager ops on this GPU (oracle port on CUDA tensors, folded weight norm)"}
    w = {k: v.to(dev) for k, v in fold_weight_norm(sd).items()}
    cfg = dict(CFG, negative_slope=0.1)
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.benchmark = True
    try:
        with torch.no_grad():
            for tag, tf32 in (("c2_fp32", False), ("c2_tf32", True)):
                torch.backends.cudnn.allow_tf32 = tf32
                torch.backends.cuda.matmul.allow_tf32 = tf32
                ms = _time_cuda(lambda: ref_ops.hifigan_generator(w, mel_dev, cfg), 5, 3, flush)
                out[tag] = {"ms_per_step": ms, "samples_per_s": BATCH * FRAMES * HOP / (ms * 1e-3)}
        # ---- C5 train step, eager autograd (train.py:200-335 restated on functional ops), fp32 (TF32 off) and TF32
        d = models.HiFiGANMultiScaleMultiPeriodDiscriminator()
        dsd = synth.synth_state_dict([(k, tuple(v.shape)) for k, v in d.state_dict().items()], 4321, 1.4)
        del d
        gw = {k: v.to(dev).requires_grad_(True) for k, v in fold_weight_norm(sd).items()}
        dw = {k: v.to(dev).requires_grad_(True) for k, v in fold_weight_norm(fold_spectral_norm_eval(dsd)).items()}
        og = torch.optim.Adam(list(gw.values()), lr=2e-4, betas=(0.5, 0.9))
        od = torch.optim.Adam(list(dw.values()), lr=2e-4, betas=(0.5, 0.9))
        melmat = torch.from_numpy(ref_ops.slaney_mel_filterbank(22050, 1024, 80, 0, 11025)).t().contiguous().to(dev)
        win = torch.hann_window(1024, device=dev)
        gen = torch.Generator().manual_seed(1000)
        c = torch.randn(16, 80, 32, generator=gen).to(dev)
        y = (torch.rand(16, 1, 8192, generator=gen) - 0.5).to(dev)

        def logmel(x):
            sp = torch.stft(x.squeeze(1), 1024, 256, 1024, win, return_complex=True)
            amp = torch.sqrt(torch.clamp(sp.real**2 + sp.imag**2, min=1e-10)).transpose(1, 2)
            return torch.log(torch.clamp(torch.matmul(amp, melmat), min=1e-10))

        def step():
            y_ = ref_ops.hifigan_generator(gw, c, cfg)
            loss = 45.0 * F.l1_loss(logmel(y_), logmel(y))
            p_ = ref_ops.hifigan_msmpd(dw, y_)
            with torch.no_grad():
                p = ref_ops.hifigan_msmpd(dw, y)
            loss = loss + ref_ops.generator_adv_loss(p_) + 2.0 * ref_ops.feature_match_loss(p_, p)
            og.zero_grad(set_to_none=True)
            od.zero_grad(set_to_none=True)
            loss.backward()
            og.step()
            with torch.no_grad():
                y_ = ref_ops.hifigan_generator(gw, c, cfg)
            real, fake = ref_ops.discriminator_adv_loss(ref_ops.hifigan_msmpd(dw, y_), ref_ops.hifigan_msmpd(dw, y))
            od.zero_grad(set_to_none=True)
            (real + fake).backward()
            od.step()

        for tag, tf32 in (("c5_step_fp32", False), ("c5_step_tf32", True)):
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cuda.matmul.allow_tf32 = tf32
            ms = _time_cuda(step, 3, 2, flush)
            out[tag] = {"ms_per_step": ms, "steps_per_s": 1e3 / ms}
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = old
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the secondary train-step measurement")
    ap.add_argument("--no-eager", action="store_true", help="skip the PyTorch-eager-on-GPU side measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the audio of the last timed step to DIR/audio.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import __graft_entry__

    __graft_entry__.build()
    from parallelwavegan_b200 import capi, ops

    assert torch.cuda.is_available(), "bench.py (--impl ours) needs a CUDA device: there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        # keep stdout to the ONE JSON line: NCCL writes its version banner / debug lines to stdout unless told
        # otherwise, so whatever NCCL_DEBUG level the launcher chose goes to a per-process file instead
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        if "NCCL_DEBUG_FILE" not in os.environ:
            os.environ["NCCL_DEBUG_FILE"] = os.path.join(tempfile.gettempdir(), "bench_nccl_%h_%p.log")
        dist.init_process_group("nccl", device_id=dev)

    model, sd = synth_weights()
    model = model.to(dev)
    g = torch.Generator().manual_seed(100 + rank)
    mel_host = torch.randn(BATCH, 80, FRAMES, generator=g).pin_memory()
    mel_dev = mel_host.to(dev)
    out_host = torch.empty(BATCH, 1, FRAMES * HOP).pin_memory()
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)  # > 126 MB L2

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.no_grad():
        for _ in range(args.warmup):
            model(mel_dev)
        torch.cuda.synchronize()

        # ---- device-resident timing: K steps, per-step events, L2 flushed between steps
        sampler = ClockSampler(local_rank)
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        barrier()
        sampler.start()
        capi.reset_launch_count()
        for e0, e1 in evs:
            flush.zero_()
            e0.record()
            y = model(mel_dev)
            e1.record()
        barrier()
        launches = capi.launch_count()
        clocks = sampler.stop()
        ms = sum(e0.elapsed_time(e1) for e0, e1 in evs)
        timed_out = y.float().cpu() if args.dump_outputs else None

        # ---- end to end through the public API: pinned host mels in, host audio out, every step
        for _ in range(2):
            out_host.copy_(model(mel_host.to(dev, non_blocking=True)), non_blocking=True)
        barrier()
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            flush.zero_()
            y = model(mel_host.to(dev, non_blocking=True))
            out_host.copy_(y, non_blocking=True)
        e1.record()
        barrier()
        ms_e2e_total = e0.elapsed_time(e1)
        # subtract nothing: the flush is part of the region here (it is ~0.1 ms of a multi-ms step)

        # ---- per-kernel-class timing for the roofline (separate instrumented pass)
        ops.PROFILE = []
        for _ in range(3):
            flush.zero_()
            model(mel_dev)
        torch.cuda.synchronize()
        prof = ops.PROFILE
        ops.PROFILE = None

    # ---- self-check of the timed output: utterance 0 of the last timed step vs the CPU oracle (rank 0)
    parity = None
    if rank == 0 and not args.no_cpu_baseline:
        from oracle.ref_ops import fold_weight_norm as _fold

        ref0 = cpu_reference_forward(_fold(sd), mel_host[:1].clone())
        y0 = y[:1].float().cpu()
        rel = float((y0.double() - ref0.double()).norm() / ref0.double().norm())
        mx = float((y0.double() - ref0.double()).abs().max() / ref0.double().abs().max())
        parity = {"utterance": 0, "rel_l2_vs_oracle": rel, "max_abs_over_peak": mx, "tolerance": 1e-3}
        assert rel <= 1e-3, f"bench output does not match the oracle: rel-L2 {rel:.3e}"

    batch1 = eager_gpu = None
    try:
        batch1 = measure_batch1(model, dev, flush)
    except Exception as e:
        batch1 = {"error": repr(e)[:300]}
    if rank == 0 and not args.no_eager:
        try:
            eager_gpu = measure_torch_eager_gpu(dev, sd, mel_dev, flush)
        except Exception as e:
            eager_gpu = {"error": repr(e)[:300]}
        torch.cuda.empty_cache()
    if dist is not None:
        dist.barrier()

    train = train_pwg = None
    if not args.no_train:
        try:
            train = measure_train_step(dev, rank, local_rank, world, dist)
        except Exception as e:  # the headline line must survive a failure of the secondary measurement
            train = {"error": repr(e)[:300]}
        try:  # BASELINE.json configs[2]: per-GPU batch 64, DDP when world > 1
            train_pwg = measure_pwg_train_step(dev, rank, local_rank, world, dist)
        except Exception as e:
            train_pwg = {"error": repr(e)[:300]}
        torch.cuda.empty_cache()

    from parallelwavegan_b200 import sharding

    local_samples = BATCH * FRAMES * HOP * args.steps
    sec, samples = sharding.reduce_stats(ms * 1e-3, local_samples, device=dev, dist=dist)  # max time, sum of samples
    sec_e2e, _ = sharding.reduce_stats(ms_e2e_total * 1e-3, local_samples, device=dev, dist=dist)
    ms, ms_e2e_total = sec * 1e3, sec_e2e * 1e3
    value = samples / sec
    e2e_value = samples / sec_e2e

    # roofline of the dominant kernel class
    agg = {}
    for name, fl, by, a, b, _desc in prof:
        d = agg.setdefault(name, [0.0, 0.0, 0.0, 0])
        d[0] += fl
        d[1] += by
        d[2] += a.elapsed_time(b)
        d[3] += 1
    dom = max(agg, key=lambda k: agg[k][2])
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    tf_peak = peaks.get("bf16_tflops_sustained") or 1400.0
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)" if peaks else "fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)"
    fl, by, tms, cnt = agg[dom]
    achieved = fl / (tms * 1e-3) / 1e12
    # DRAM traffic of the dominant class: measured with ncu on the same command (launch list with dram__bytes_read/write,
    # tools/gpu/run1.sh), averaged over every launch of the class in the 16x80x400 forwards -- not a constant of one launch
    traffic, traffic_note = None, "no ncu launch list committed for this build"
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic_r2_bench.json")))["dominant_class_batch16"]
        if tj["kernel"].startswith(dom):
            traffic = tj["dram_bytes_per_launch"]
            traffic_note = (f"mean dram__bytes_read.sum + dram__bytes_write.sum per launch over {tj['launches_counted']} launches of the class "
                            f"(ncu launch list of `bench.py --steps 1 --warmup 3`, profiles/traffic_r2_bench.json); the class's share of the forward "
                            f"under ncu is {tj['time_share_of_forward_under_ncu']:.3f}")
    except Exception:
        pass
    alg_bytes_per_launch = by / cnt
    roofline = {"kernel": dom, "bound": "tensor", "achieved": achieved, "peak": tf_peak, "unit": "TFLOP/s",
                "frac": achieved / tf_peak, "traffic": traffic, "traffic_note": traffic_note,
                "algorithmic_bytes_per_launch": alg_bytes_per_launch, "algorithmic_flops_per_launch": fl / cnt,
                "peak_source": peak_src,
                "launches_per_step": cnt / 3, "avg_launch_ms": tms / cnt, "share_of_step": tms / sum(v[2] for v in agg.values()),
                "algorithmic_flops_per_step": fl / 3,
                "note": "achieved = algorithmic conv FLOPs (2*MAC, fp32 semantics) / summed CUDA-event durations of the class; the kernel issues 3 bf16 MMAs per algorithmic MAC (bf16x3 split for fp32 parity), so frac <= 1/3 by construction"}

    if args.dump_outputs:
        import numpy as np

        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "audio.npy" if world == 1 else f"audio_rank{rank}.npy"), timed_out.numpy())

    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline:
            from oracle.ref_ops import fold_weight_norm

            wf = fold_weight_norm(sd)
            cores, host_cores = tune_cpu_threads(wf)
            sb = 4
            v, dt = time_cpu(wf, sb, FRAMES, 2)
            cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": f"{sb} of the {BATCH} utterances (80x{FRAMES} mels each), decoded utterance by utterance like the --impl reference arm "
                             f"(bin/decode.py:214-243), best of 2, {dt:.2f} s, oracle port (torch CPU fp32 ATen ops), "
                             f"{cores} threads = best of a probe over 8..{host_cores} on a {host_cores}-core host"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": shared_config(world),
            "precision": "fp32 I/O and accumulation; wide convs on tcgen05 with a bf16x3 operand split (parity measured below)",
            "l2": "flushed between timed steps (256 MiB write); activations (>=210 MB per stage tensor) exceed L2 anyway",
            "parity": parity,
            "batch1": batch1,
            "torch_eager_gpu": eager_gpu,
            "rtf": FS / (value / world) , "x_realtime_per_gpu": (value / world) / FS,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": mel_host.numel() * 4 * world,
                    "d2h_bytes_per_step": out_host.numel() * 4 * world, "ms_per_step": ms_e2e_total / args.steps},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": roofline,
            "cpu_baseline": cpu,
            "train": train,
            "train_pwg": train_pwg,
            "kernel_classes": {k: {"ms_per_step": v[2] / 3, "launches_per_step": v[3] / 3, "tflops": v[0] / (v[2] * 1e-3) / 1e12,
                                   "alg_GBps": v[1] / (v[2] * 1e-3) / 1e9} for k, v in agg.items()},
        }
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
