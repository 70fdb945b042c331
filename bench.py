#!/usr/bin/env python
"""bench.py -- BASELINE.json metric: audio frames/sec (22.05 kHz) of the generator forward.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A "step" is one generator forward over one synthetic batch of config 2 (B=64 mel segments of
80 x 32 frames -> 64 x 8192 audio frames) per GPU.  1 audio frame = 1 PCM sample; 1 mel frame = 256
audio frames (SURVEY 8d).  Weights are seeded random-init (melgan_multi_b200.synth), data synthetic.

  value      device-resident throughput: mel already in HBM, CUDA events around the C-ABI
             device-pointer call (mg_gen_forward), L2 flushed between steps, max over ranks.
  e2e        the same metric through the host-buffer C ABI (mg_gen_engine_forward): pinned host mel
             in, H2D copy, kernels, D2H copy of the audio out, every step, wall clock, max over ranks.
  roofline   dominant kernel (stage 1: ConvT 256->128 + 128-channel ResBlock, 44% of the FLOPs),
             per-kernel CUDA events from mg_gen_forward_timed in a second pass of K steps.
  cpu_baseline  oracle/torch_port.generator_forward_reference (the reference's forward on PyTorch-CPU/oneDNN,
             per-forward weight-norm included, all host threads) on the FULL config-2 batch, a bounded
             number of iterations, median; rank 0 at N=1 only.
  --impl reference   times that same CPU port as the reference arm at the same config (the reference is pure
             Python and /root/reference does not exist on the GPU box); value from the MEDIAN step.
  --dump-outputs DIR   writes what the timed path returned in its last timed step, rank 0's [64, 1, 8192] fp32 audio
             (2 MB), to DIR/audio.npy.  Weights and mel inputs are seeded, so runs with the same arguments see the
             same inputs and two builds can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

B_PER_GPU, T_FRAMES = 64, 32
METRIC = "generator_fwd_audio_frames_per_sec"
UNIT = "audio_frames/s"
WORKLOAD = "configs[1]: Generator forward, batch=64, 80x32 mel -> 64x8192 samples, fp32"


def flops_per_mel_frame():
    pre = 2 * 80 * 512 * 7
    stages = []
    for i, (cin, cout, s) in enumerate([(512, 256, 8), (256, 128, 8), (128, 64, 2), (64, 32, 2)]):
        up = [8, 64, 128, 256][i]
        stages.append(up * (2 * 2 * cin * cout) + up * 6 * (2 * cout * cout * 3))
    post = 2 * 32 * 7 * 256
    return pre, stages, post


ALG_BYTES_PER_FRAME = 152896  # SURVEY 8(d): per-stage-fused design, fp32 activations in/out of each kernel
ALG_WEIGHT_BYTES = 18080000   # SURVEY 8(d): 18.08 MB of folded weights + biases, read once per launch chain
STAGE_BYTES_PER_FRAME = [320 * 1 + 2048, 2048 + 8192, 8192 + 32768, 32768 + 32768, 32768 + 1024]


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained"), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """Samples SM clock and clock-event (throttle) reasons of one GPU WHILE the timed region runs: an in-process NVML
    poller thread (2 ms period; the main thread sits in ctypes/CUDA calls that release the GIL).  nvidia-smi -lms is the
    fallback, but its ~1 s start-up and >=100 ms period see at most one sample of a 25 ms timed region."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index):
        import threading
        self.samples, self.mask, self.max_mhz, self._stop = [], 0, None, False
        self.smi = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical devices; honour CUDA_VISIBLE_DEVICES if it is a plain index list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = index
            if vis and all(v.strip().isdigit() for v in vis.split(",")) and index < len(vis.split(",")):
                phys = int(vis.split(",")[index])
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nv = pynvml

            def poll():
                while not self._stop:
                    try:
                        self.samples.append(float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
                        self.mask |= int(self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                    except Exception:
                        pass
                    time.sleep(0.002)
            self.t = threading.Thread(target=poll, daemon=True)
            self.t.start()
        except Exception:
            self.nv = None
            self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                 "clocks_event_reasons.sw_power_cap")
            try:
                self.smi = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + q,
                                             "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                            stderr=subprocess.DEVNULL)
            except OSError:
                self.smi = None

    def mark(self):
        """Call right before the timed region: only later samples count."""
        self.samples, self.mask = [], 0

    def stop(self):
        if self.nv is not None:
            self._stop = True
            self.t.join(timeout=1)
            if not self.samples:
                return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["no samples"], "source": "nvml"}
            hi = [c for c in self.samples if c >= 0.5 * max(self.samples)]
            return {"sm_mhz": statistics.median(hi), "sm_max_mhz": self.max_mhz,
                    "reasons": sorted(n for bit, n in self.REASONS.items() if self.mask & bit),
                    "samples": len(self.samples), "source": "nvml poll, 2 ms"}
        if self.smi is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.smi.terminate()
        try:
            self.smi.wait(timeout=5)
        except Exception:
            self.smi.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            if len(r) < 8:
                continue
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except ValueError:
                continue
            for n, v in zip(names, r[4:8]):
                if v.strip() == "Active":
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"], "source": "nvidia-smi"}
        hi = [c for c in sm if c >= 0.5 * max(sm)]
        return {"sm_mhz": statistics.median(hi), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvidia-smi -lms 100"}


def usable_cpus():
    """Host threads this process may really use: min(affinity mask, cgroup v2 cpu.max quota).  os.cpu_count()
    alone reports the machine (128 on the GPU boxes) while the container is capped (16), and oneDNN with 128
    threads on a 16-CPU quota runs ~500x slower."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return max(1, n)


def cpu_port_steps(n_steps, warmup, budget_s=None):
    """Times oracle/torch_port.generator_forward_reference (weight-norm fold of the 30 layers + the conv graph: what the
    reference's Generator.forward does on a CPU) on the whole config-2 batch, all usable host threads.  Returns
    (per-step seconds list, cores).  budget_s bounds the timed part (at least 2 steps)."""
    import torch
    from melgan_multi_b200 import synth
    from oracle import torch_port
    cores = usable_cpus()
    torch.set_num_threads(cores)
    params = torch_port.reference_state(synth.generator_state(1234))
    xs = [torch.from_numpy(synth.mel_input(B_PER_GPU, T_FRAMES, i)) for i in range(2)]
    for i in range(warmup):  # oneDNN primitive creation + thread-pool spin-up take several calls
        torch_port.generator_forward_reference(params, xs[i % 2])
    times, t_all = [], time.perf_counter()
    for i in range(n_steps):
        t0 = time.perf_counter()
        torch_port.generator_forward_reference(params, xs[i % 2])
        times.append(time.perf_counter() - t0)
        if budget_s is not None and len(times) >= 2 and time.perf_counter() - t_all > budget_s:
            break
    return times, cores


def run_reference(args):
    """Reference arm: the reference's CPU implementation of the path (PyTorch-CPU restatement of models.py:61-71 with the
    per-forward weight-norm hooks), same config as the B200 arm: the full B=64 batch per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    times, cores = cpu_port_steps(args.steps, max(3, args.warmup))
    frames = B_PER_GPU * T_FRAMES * 256
    med = statistics.median(times)
    val = frames / med
    sample = ("the whole config-2 batch (64 x 80x32 mel) per step; PyTorch-CPU (oneDNN) restatement of the reference forward "
              "incl. its 30 per-forward weight-norm folds, %d threads; value = frames / MEDIAN step (mean %.3f s, min %.3f s, "
              "max %.3f s over %d steps)" % (cores, sum(times) / len(times), min(times), max(times), len(times)))
    emit(({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": len(times), "warmup": max(3, args.warmup), "ms_per_step": 1e3 * med,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "batch_per_gpu": B_PER_GPU, "mel_frames": T_FRAMES, "global_batch": B_PER_GPU,
                   "timing": "median of per-step wall clock", "weights": "seeded random init"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def multi_gpu_blocks(dev, rank, world, barrier, max_over_ranks, steps=10, warmup=3):
    """Extra keys of the JSON line when WORLD_SIZE > 1 (the headline metric is unchanged): the two paths of SURVEY 8(e)
    that DO talk to other ranks, measured with CUDA events under barriers, max over ranks.
      ddp_train_step   BASELINE config 4: one train.py:108-129 step (G-step + D-step, losses, backward, multi-tensor Adam) at
                       batch 16 x 8192 samples per GPU through melgan_multi_b200.distributed over NCCL, against the same step
                       without any communication and against the bare all-reduces of the two gradient buffers.
      utterance_shard  BASELINE config 5 cut along TIME over the ranks (8-frame halo, no data-path collective, one
                       all_gather of the audio) against the whole utterance on one GPU."""
    import torch
    import torch.distributed as dist
    from melgan_multi_b200 import distributed as mgd
    from melgan_multi_b200 import models, synth
    from melgan_multi_b200.optim import Adam

    def build():
        gen = models.Generator()
        gen.load_state_dict({k: torch.from_numpy(v) for k, v in synth.generator_state(1234).items()})
        msd = models.MultiScaleDiscriminator()
        msd.load_state_dict({k: torch.from_numpy(v) for k, v in synth.discriminator_state(4321).items()})
        return gen.to(dev).train(), msd.to(dev).train()

    x = torch.from_numpy(synth.mel_input(16, 32, 100 + rank)).to(dev)
    y = torch.from_numpy(synth.audio_input(16, 8192, 200 + rank)).to(dev)

    def train_step(gen, msd, g_opt, d_opt, comm):
        g_opt.zero_grad()
        y_ghat = gen(x)
        dr, dg, fr, fg = msd(y, y_ghat)
        loss_gen = models.generator_loss(dg) + models.feature_loss(fr, fg)
        if comm:
            mgd.reduce_tensor(loss_gen.data, world)  # train.py:113-114 (logging all-reduce; the .item() sync is left out)
        loss_gen.backward()
        g_opt.step()
        d_opt.zero_grad()
        dr, dg, _, _ = msd(y, y_ghat.detach())
        loss_disc, _, _ = models.discriminator_loss(dr, dg)
        if comm:
            mgd.reduce_tensor(loss_disc.data, world)
        loss_disc.backward()
        d_opt.step()
        return loss_gen, loss_disc

    def timed(fn, n, w):
        for _ in range(w):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1) / n)

    out = {}
    # -- same step, no communication (unwrapped replicas): the compute floor
    gen0, msd0 = build()
    g0, d0 = Adam(gen0.parameters(), 2e-4, betas=(0.5, 0.9)), Adam(msd0.parameters(), 2e-4, betas=(0.5, 0.9))
    nocomm_ms = timed(lambda: train_step(gen0, msd0, g0, d0, False), steps, warmup)
    del gen0, msd0, g0, d0
    # -- data-parallel step
    gen1, msd1 = build()
    mgd.apply_gradient_allreduce(gen1)
    mgd.apply_gradient_allreduce(msd1)
    g1, d1 = Adam(gen1.parameters(), 2e-4, betas=(0.5, 0.9)), Adam(msd1.parameters(), 2e-4, betas=(0.5, 0.9))
    ddp_ms = timed(lambda: train_step(gen1, msd1, g1, d1, True), steps, warmup)
    sg, sd = dict(gen1._grad_reducer.stats), dict(msd1._grad_reducer.stats)
    # the same wrapped step with the collectives themselves left out (hooks, bucket adoption, /world still run): what is left of
    # ddp_ms - dry_ms is communication that backward did not hide
    gen1._grad_reducer.dry = msd1._grad_reducer.dry = True
    dry_ms = timed(lambda: train_step(gen1, msd1, g1, d1, False), steps, warmup)
    gen1._grad_reducer.dry = msd1._grad_reducer.dry = False
    passes = max(1, sg["passes"])
    bytes_step = (sg["allreduce_bytes"] + sd["allreduce_bytes"]) / passes
    skipped_step = sd["skipped_bytes"] / passes
    # -- the bare collectives of one step: G's 18.1 MB buffer once, D's three per-Discriminator buckets once
    fg_, fd_ = gen1._grad_reducer, msd1._grad_reducer

    def bare():
        ws = [dist.all_reduce(fg_.flat, async_op=True)]
        for s_, e_, _m in fd_.buckets:
            ws.append(dist.all_reduce(fd_.flat.narrow(0, s_, e_ - s_), async_op=True))
        for w_ in ws:
            w_.wait()
    bare_ms = timed(bare, 20, 5)
    gbytes, dbytes = fg_.flat.numel() * 4, fd_.flat.numel() * 4
    exposed = max(0.0, ddp_ms - dry_ms)
    out["ddp_train_step"] = {
        "config": "configs[3]: DDP train step batch=16/gpu, 8192-sample segments, %d x B200, NCCL all-reduce" % world,
        "ms": ddp_ms, "ms_same_step_unwrapped_single_gpu": nocomm_ms, "ms_wrapped_without_the_collectives": dry_ms,
        "exposed_communication_ms": exposed,
        "allreduce_ms": bare_ms,
        "overlap_frac": (sg["bytes_launched_with_backward_left"] + sd["bytes_launched_with_backward_left"]) /
                        max(1, sg["allreduce_bytes"] + sd["allreduce_bytes"]),
        "overlap_frac_definition": "share of all-reduced gradient bytes whose collective was launched (from a gradient hook) "
                                   "while autograd still had gradients to produce, i.e. with backward compute left to overlap; the "
                                   "measured cost is exposed_communication_ms = ms - ms_wrapped_without_the_collectives (includes "
                                   "the two synchronous logging all-reduces of train.py:113,124 and SM contention of the NCCL kernels)",
        "bytes": bytes_step, "bytes_reference_would_send": gbytes + 2 * dbytes, "bytes_skipped_per_step": skipped_step,
        "segments_per_s": 16 * world / (ddp_ms * 1e-3),
        "allreduce_busbw_gbs": 2 * (world - 1) / world * (gbytes + dbytes) / (bare_ms * 1e-3) / 1e9,
        "buckets_bytes": {"G": [(e_ - s_) * 4 for s_, e_, _m in fg_.buckets], "D": [(e_ - s_) * 4 for s_, e_, _m in fd_.buckets]},
        "limiting_collective": "all-reduce of the discriminators' gradients: 3 buckets of 22.6 MB (one per Discriminator, "
                               "21 MB of each is conv_post1's 1024x1024x5 weight_v), launched as each scale's backward ends; "
                               "the generator's 18.1 MB bucket is launched when its (single-node) backward returns",
        "dedup": "discriminator gradients of the generator step (67.7 MB) are not reduced: learned at run time from the "
                 "optimizer/forward order, no train.py edit",
        "steps": steps, "warmup": warmup, "dtype": "f32 (forwards: 3-pass split-bf16 tcgen05; backward: see DESIGN.md)",
    }
    del gen1, msd1, g1, d1
    # -- config 5 sharded along time
    gen, _ = build()
    gen.eval()
    mel = torch.from_numpy(synth.mel_input(1, 1000, 0)).to(dev)
    with torch.no_grad():
        whole_ms = timed(lambda: gen(mel), 20, 5)
        shard_ms = timed(lambda: mgd.generate_sharded(gen, mel, gather=False), 20, 5)
        gather_ms = timed(lambda: mgd.generate_sharded(gen, mel, gather=True), 20, 5)
    out["utterance_shard"] = {
        "config": "configs[4]: long-utterance inference, batch=1, 80x1000 mel, cut along time over %d GPUs (8-frame halo)" % world,
        "ms_one_gpu_whole_utterance": whole_ms, "ms_sharded": shard_ms, "ms_sharded_with_all_gather": gather_ms,
        "speedup": whole_ms / shard_ms, "efficiency": whole_ms / shard_ms / world,
        "collective": "none on the data path; optional all_gather of 256 000 fp32 samples",
        "note": "one utterance is bound by the latency of a tile's six dependent convs, not by throughput: sharding time "
                "shortens each rank's grid, not the per-tile chain",
    }
    return out


_JSON_OUT = None


def claim_stdout():
    """stdout must carry exactly ONE JSON line, but libraries write there too (NCCL prints its version banner to fd 1
    whatever NCCL_DEBUG_FILE says): keep a private copy of the real stdout for the result and point fd 1 at stderr."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(obj):
    _JSON_OUT.write(json.dumps(obj) + "\n")
    _JSON_OUT.flush()


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-budget", type=float, default=15.0, help="seconds of CPU-baseline timing")
    ap.add_argument("--no-multi", action="store_true", help="skip the DDP train-step / utterance-shard blocks at N > 1")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the audio of the last timed step (rank 0) to DIR/audio.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the output of the b200 path")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from melgan_multi_b200 import engine, synth

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # stdout carries exactly one JSON line: NCCL's own banner / debug log (stdout by default) goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    K, W, B, T = args.steps, args.warmup, B_PER_GPU, T_FRAMES
    peaks = load_peaks()
    state = synth.generator_state(1234)

    # ---- device-resident path -----------------------------------------------------------
    gd = engine.GeneratorDevice(dev)
    order = [n for n, *_ in synth.GENERATOR_LAYERS]
    to = lambda a: torch.from_numpy(a).to(dev)
    gd.pack([to(state[n + ".weight_v"]) for n in order], [to(state[n + ".weight_g"]) for n in order],
            [to(state[n + ".bias"]) for n in order])
    mels = [to(synth.mel_input(B, T, 10 * rank + i)) for i in range(4)]
    out = torch.empty((B, 1, 256 * T), dtype=torch.float32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    sampler = ClockSampler(local_rank)
    for i in range(W):
        flush.zero_()
        gd.forward(mels[i % 4], out)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    barrier()
    sampler.mark()
    for k in range(K):
        flush.zero_()
        ev[k][0].record()
        gd.forward(mels[k % 4], out)
        ev[k][1].record()
    barrier()
    # the passes below reuse `out`: keep the last timed step's result now
    last_audio = out.cpu().numpy() if args.dump_outputs and rank == 0 else None
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = max_over_ranks(sum(step_ms))
    frames_per_step = B * T * 256 * world
    value = K * frames_per_step / (total_ms * 1e-3)

    # ---- per-kernel pass (roofline) -------------------------------------------------------
    names, kms = None, None
    for k in range(K):
        flush.zero_()
        timed = gd.forward_timed(mels[k % 4], out)
        if names is None:
            names, kms = [n for n, _ in timed], np.zeros(len(timed))
        kms += np.array([v for _, v in timed])
    kms /= K
    clocks = sampler.stop()
    pre_f, stage_f, post_f = flops_per_mel_frame()
    frames = B * T
    up_f = [[8, 64, 128, 256][i] * (2 * 2 * cin * cout) * frames
            for i, (cin, cout) in enumerate([(512, 256), (256, 128), (128, 64), (64, 32)])]
    res_f = [stage_f[i] * frames - up_f[i] for i in range(4)]
    flops_of = {"conv_pre": pre_f * frames, "post": post_f * frames}
    for i in range(4):
        flops_of["up%d" % i] = up_f[i]
        flops_of["res%d" % i] = res_f[i]
        flops_of["stage%d(up+res)" % i] = up_f[i] + res_f[i]
    flops_of["stage3(up+res+post)"] = up_f[3] + res_f[3] + post_f * frames
    flops_of["res3+post"] = res_f[3] + post_f * frames
    flops_of["up2+res2"] = up_f[2] + res_f[2]  # stride-2 ConvT fused at the front of the stage kernel
    flops_of["up3+res3+post"] = up_f[3] + res_f[3] + post_f * frames
    for i in range(3):  # the next stage's ConvT fused at the tail of ResBlock i's kernel (the default chain)
        flops_of["res%d+up%d" % (i, i + 1)] = res_f[i] + up_f[i + 1]
    k_flops = [flops_of[n] for n in names]
    dom = [i for i, n in enumerate(names) if n.startswith("res1")][0]
    dom_name = names[dom]
    dom_tflops = k_flops[dom] / (kms[dom] * 1e-3) / 1e12
    fwd_flops = sum(k_flops)
    packed_bytes = engine.lib().mg_gen_packed_bytes()
    # ALGORITHMIC HBM bytes = SURVEY 8(d): 152 896 B per mel frame (per-stage-fused design) + 18.08 MB of folded fp32 weights
    # = 331.2 MB at config 2.  What this pipeline's kernels actually move by design is more: the ConvT outputs of the
    # stages whose ConvT is a separate kernel make one extra HBM round trip (written by up_i, re-read by res_i), and the
    # weights are streamed as split-bf16 (hi + lo: the same 4 bytes per weight) -- reported as moved_bytes / wasted ratio.
    # per mel frame, fp32: every kernel boundary of the chain is one write + one read of the tensor that crosses it
    boundary = {"conv_pre": 2048, "up0": 8192, "res0": 8192, "up1": 32768, "res0+up1": 32768, "res1": 32768, "up2": 32768,
                "res1+up2": 32768, "res2": 32768, "up2+res2": 32768, "up3": 32768, "res2+up3": 32768}
    moved_frame = 320 + 1024 + 2 * sum(boundary[n] for n in names if n in boundary)
    extra = moved_frame - ALG_BYTES_PER_FRAME
    alg_bytes = ALG_BYTES_PER_FRAME * frames + ALG_WEIGHT_BYTES
    moved_bytes = (ALG_BYTES_PER_FRAME + extra) * frames + packed_bytes
    fwd_ms = total_ms / K
    # dram bytes per launch of the dominant kernel from the committed `ncu --set full` capture -- quoted only if that capture
    # was taken with the kernel configuration this build runs (profiles/r02_ncu_traffic.json records mg_gen_kernel_config)
    traffic, traffic_note = None, None
    L_ = engine.lib()
    L_.mg_gen_kernel_config.restype = ctypes.c_char_p
    L_.mg_gen_kernel_config.argtypes = [ctypes.c_int, ctypes.c_int]
    cfg_now = L_.mg_gen_kernel_config(dom, T).decode()
    tpath = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
    if os.path.exists(tpath):
        t = json.load(open(tpath)).get(dom_name)
        if t and t.get("kernel_config") == cfg_now:
            traffic = t["dram_read_bytes"] + t["dram_write_bytes"]
            traffic_note = ("dram__bytes_read.sum + dram__bytes_write.sum of one launch, ncu --set full of this kernel configuration "
                            "(profiles/r02_ncu_traffic.json, %.1f us under ncu); algorithmic HBM bytes of this kernel: 2 * 64*128*2048*4 "
                            "= 134.2 MB (the 126 MB L2 keeps part of the output)" % t["gpu_time_us"])
        else:
            traffic_note = ("STALE CAPTURE IGNORED: profiles/r02_ncu_traffic.json holds %r for %s, this build runs %r -- re-run "
                            "scripts/gpu_profile_r02.sh" % (t.get("kernel_config") if t else None, dom_name, cfg_now))
            print("bench.py: " + traffic_note, file=sys.stderr)
    else:
        traffic_note = "no ncu capture committed for this build"
    roofline = {
        "kernel": ("resblock_tc_kernel<C=128> (%s: stage-1 ResBlock, 6 k3 convs%s; %.0f%% of generator FLOPs)" % (
            dom_name, " + stage-2 ConvTranspose at its tail" if "+" in dom_name else "", 100.0 * k_flops[dom] / sum(k_flops))),
        "bound": "tensor", "achieved": dom_tflops, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
        "frac": dom_tflops / peaks["bf16_tflops"], "traffic": traffic,
        "traffic_note": traffic_note, "kernel_config": cfg_now,
        "peak_source": "%s bf16 dense burst (MEASURED_PEAKS.json)" % peaks["source"],
        "algorithmic_flops_per_launch": k_flops[dom], "avg_launch_ms": float(kms[dom]),
        "math": ("split-bf16 tcgen05: 3 MMA passes per product, so tensor-pipe work is 3x the algorithmic FLOPs "
                 "(pipe-level fraction = 3 * frac)"),
        "kernel_ms": {n: float(v) for n, v in zip(names, kms)},
        "kernel_tflops": {n: k_flops[i] / (kms[i] * 1e-3) / 1e12 for i, n in enumerate(names)},
        "hbm": {"achieved": alg_bytes / (fwd_ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": alg_bytes / (fwd_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                "algorithmic_bytes_per_forward": alg_bytes, "moved_bytes_per_forward_by_design": moved_bytes,
                "wasted_traffic_ratio": moved_bytes / alg_bytes,
                "note": "whole forward, SURVEY 8(d) bytes (152 896 B/frame + 18.08 MB weights); the fused generator is "
                        "683 FLOP/B, i.e. math-bound: 60 % of HBM peak would need 2.5 PFLOP/s (SURVEY 8d)"},
        "forward_tflops": fwd_flops / (fwd_ms * 1e-3) / 1e12,
    }

    # ---- end to end through the host-buffer C ABI -----------------------------------------
    host = engine.GeneratorHost(B, T)
    host.load_state(state)
    pin_in = [torch.from_numpy(synth.mel_input(B, T, 10 * rank + i)).pin_memory() for i in range(4)]
    pin_out = torch.empty((B, 1, 256 * T), dtype=torch.float32).pin_memory()
    for i in range(W):
        host.forward_ptr(pin_in[i % 4].data_ptr(), pin_out.data_ptr(), B, T)
    barrier()
    t0 = time.perf_counter()
    for k in range(K):
        host.forward_ptr(pin_in[k % 4].data_ptr(), pin_out.data_ptr(), B, T)
    e2e_s = time.perf_counter() - t0
    barrier()
    checksum = float(pin_out.double().abs().sum())
    e2e_s = max_over_ranks(e2e_s)
    e2e_value = K * frames_per_step / e2e_s
    host.close()

    cpu = None
    if rank == 0 and world == 1:
        times, cores = cpu_port_steps(50, 3, args.cpu_budget)
        med = statistics.median(times)
        cpu = {"value": B * T * 256 / med, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": "the whole config-2 batch (64 x 80x32 mel), %d iterations, median %.3f s; oracle/torch_port."
                         "generator_forward_reference = the reference forward (incl. per-forward weight-norm) on "
                         "PyTorch-CPU/oneDNN, all threads" % (len(times), med)}

    multi = multi_gpu_blocks(dev, rank, world, barrier, max_over_ranks) if world > 1 and not args.no_multi else None

    if last_audio is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "audio.npy"), last_audio)
    if rank == 0:
        emit(({
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 in/out; products as 3 split-bf16 tcgen05 passes with fp32 accumulation (fp32-equivalent, ~1e-5)",
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "batch_per_gpu": B, "mel_frames": T, "global_batch": B * world,
                       "parallelism": "dp%d (independent batches, no collective)" % world,
                       "l2": "flushed between steps (256 MiB memset)", "weights": "seeded random init"},
            "mel_frames_per_s": value / 256, "realtime_factor": value / 22050.0,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": B * 80 * T * 4 * world,
                    "d2h_bytes_per_step": B * 256 * T * 4 * world, "ms_per_step": 1e3 * e2e_s / K,
                    "api": "mg_gen_engine_forward (host buffers, pinned)", "output_abs_sum": checksum},
            "gpu_launches": K * world * engine.lib().mg_gen_forward_launches() * engine.lib().mg_gen_forward_slices(B, T),
            "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks,
            **({"multi_gpu": multi} if multi else {}),
        }))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
