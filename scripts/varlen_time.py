"""Ragged generator batches (mg_gen_forward_varlen) against the ways a caller without per-item lengths would vocode them.

Workloads (seeded):
  S  B = 64: 32 lengths drawn from [8, 56] plus their mirrors 64 - v, i.e. exactly 2048 mel frames -- the frames of BASELINE
     config 2 (64 x 32), so the same-frames arm IS config 2
  U  B = 16 utterances of 100..1000 frames (a TTS batch of long sentences)
Arms:
  varlen      one call, Generator(x, lengths)
  padded      one uniform call on the batch padded to Tmax (the audio past each end is wrong and must be trimmed)
  per_item    one uniform call per item, back to back on the stream
  same_frames one uniform batch with the same total frames (S: 64 x 32; U: 16 x round(frames / 16))
Every step is one call of one arm between two CUDA events, with the L2 (126 MB) overwritten by a 256 MB memset before it;
arms alternate within a round, the median of the steps is reported.  Also checks that the varlen outputs equal the
per-item loop's bit for bit on the timed inputs, and records the card name and power limit.
usage: python scripts/varlen_time.py [--steps 30] [--out profiles/r03_varlen_time.json]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from melgan_multi_b200 import models, synth  # noqa: E402


def workloads():
    rs = np.random.RandomState(2048)
    v = rs.randint(8, 57, size=32)
    s = np.concatenate([v, 64 - v])
    rs.shuffle(s)
    u = np.random.RandomState(1000).randint(100, 1001, size=16)
    return {"S": s, "U": u}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], stdout=subprocess.PIPE, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001 -- the measurement stands without it, the record says why
        q = "nvidia-smi unavailable: %s" % e
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join("profiles", "r03_varlen_time.json"))
    a = ap.parse_args()
    assert a.steps >= 20, "the median wants >= 20 steps"
    if not torch.cuda.is_available():
        raise SystemExit("varlen_time.py measures on the GPU; no CUDA device here")
    g = models.Generator()
    g.load_state_dict({k: torch.from_numpy(v) for k, v in synth.generator_state(1234).items()})
    g = g.cuda().eval()
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")  # 256 MB > L2
    rec = {"card": card(), "steps": a.steps, "l2_flush_bytes": flush.numel() * 4, "statistic": "median device ms per call",
           "workloads": {}}
    with torch.no_grad():
        for name, lengths in workloads().items():
            lengths = [int(n) for n in lengths]
            B, T, frames = len(lengths), max(lengths), sum(lengths)
            x = torch.from_numpy(synth.mel_input(B, T, 7)).cuda()
            items = [x[b:b + 1, :, :n].contiguous() for b, n in enumerate(lengths)]
            su = (64, 32) if name == "S" else (B, round(frames / B))
            xu = torch.from_numpy(synth.mel_input(su[0], su[1], 8)).cuda()
            arms = {
                "varlen": lambda: g(x, lengths=lengths),
                "padded": lambda: g(x),
                "per_item": lambda: [g(it) for it in items],
                "same_frames": lambda: g(xu),
            }
            y = g(x, lengths=lengths)
            g._dev.check_status(B, T)
            equal = all(torch.equal(y[b:b + 1, :, :256 * n], g(items[b])) and not y[b, :, 256 * n:].any().item()
                        for b, n in enumerate(lengths))
            for _ in range(a.warmup):
                for fn in arms.values():
                    fn()
            ms = {k: [] for k in arms}
            for _ in range(a.steps):
                for k, fn in arms.items():
                    flush.zero_()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    fn()
                    e1.record()
                    e1.synchronize()
                    ms[k].append(e0.elapsed_time(e1))
            med = {k: float(np.median(v)) for k, v in ms.items()}
            rec["workloads"][name] = {
                "B": B, "T_max": T, "frames": frames, "lengths": lengths, "same_frames_shape": list(su),
                "median_ms": med, "spread_ms": {k: [float(min(v)), float(max(v))] for k, v in ms.items()},
                "varlen_equals_per_item": bool(equal),
                "varlen_faster_than_padded": med["varlen"] < med["padded"],
                "varlen_faster_than_per_item": med["varlen"] < med["per_item"],
                "varlen_over_same_frames": med["varlen"] / med["same_frames"],
                "varlen_M_frames_per_s": frames / med["varlen"] / 1e3,
            }
    line = json.dumps(rec)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")
    print(line)
    ok = all(w["varlen_equals_per_item"] and w["varlen_faster_than_padded"] and w["varlen_faster_than_per_item"]
             for w in rec["workloads"].values())
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
