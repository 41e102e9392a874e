#!/usr/bin/env python
"""Ragged batches on one GPU: RaggedPipeline against today's per-clip alternative and against CapturedPipeline.

    python tools/bench_ragged.py [--reps 10] [--precision fp16x3] [--out profiles/r3/bench_ragged.json]

  (a) RaggedPipeline on a seeded mix of 32 clips of 4-12 s, one replay per batch
  (b) the same 32 clips one by one, each through a CapturedPipeline built for its exact length (batch 1)
  (c) the equal-length BASELINE batch (32 x 10 s): RaggedPipeline vs CapturedPipeline per call (host staging included)
      and as graph replays alone on inputs staged beforehand, i.e. the device cost of the limits

Every timed unit is a CUDA-event interval preceded by a 256 MB write that evicts the 126 MB L2; every shape is warmed
up first and the arms alternate per repetition.  Reports emitted motion frames per second and the padding efficiency
(emitted frames / (clips x windows x 60)), with the card's name and power limit, as one JSON document.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        q = torch.cuda.get_device_name() + ", power limit unknown"
    return q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--precision", default="fp16x3")
    ap.add_argument("--clips", type=int, default=32)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_ragged.py measures the GPU: no CUDA device"
    from oracle.weights import synth_audio
    from pantomatrix_b200.emage_audio import engine as E
    from pantomatrix_b200.pipeline import CapturedPipeline, RaggedPipeline
    from synthetic_models import build_product
    E.set_precision(args.precision)
    model, vqm = build_product(seed=0, device="cuda")
    rng = np.random.default_rng(2026)
    lens = [int(n) for n in rng.integers(4 * 16000, 12 * 16000 + 1, args.clips)]
    audios = [torch.from_numpy(synth_audio(1, n, 7 + i))[0].cuda() for i, n in enumerate(lens)]
    base = torch.from_numpy(synth_audio(args.clips, 160000, 1234)).cuda()
    base_list = list(base)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def timed(fn):
        flush.fill_(1)                                 # evict L2 (126 MB) between timed units
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        return a.elapsed_time(b) / 1e3

    ragged = RaggedPipeline(model, vqm, batch=args.clips, max_samples=12 * 16000)
    per_len = {n: CapturedPipeline(model, vqm, 1, n) for n in sorted(set(lens))}
    ragged_eq = RaggedPipeline(model, vqm, batch=args.clips, max_samples=160000)     # same capacity as `captured`
    captured = CapturedPipeline(model, vqm, args.clips, 160000)
    plan = ragged.plan(lens)
    emitted = int(plan.out_len.sum())
    base_frames = args.clips * (160000 * 30 // 16000)

    arms = {
        "a_ragged_mix": lambda: ragged(audios),
        "b_one_by_one_mix": lambda: [per_len[n](a[None]) for n, a in zip(lens, audios)],
        "c_ragged_equal": lambda: ragged_eq(base_list),
        "c_captured_equal": lambda: captured(base),
        "c_ragged_replay": ragged_eq.replay,          # inputs staged by ragged_eq.load() below and by c_ragged_equal
        "c_captured_replay": captured.graph.replay,
    }
    ragged_eq.load(base_list)
    captured(base)
    for fn in arms.values():                           # warm-up of every shape
        fn(), fn()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for r in range(args.reps):
        for k in (list(arms) if r % 2 == 0 else list(arms)[::-1]):
            times[k].append(timed(arms[k]))
    frames = {"a_ragged_mix": emitted, "b_one_by_one_mix": emitted, "c_ragged_equal": base_frames,
              "c_captured_equal": base_frames, "c_ragged_replay": base_frames, "c_captured_replay": base_frames}
    res = {"card": card(), "precision": args.precision, "clips": args.clips, "reps": args.reps,
           "mix_seconds": [round(n / 16000, 3) for n in lens], "mix_emitted_frames": emitted,
           "mix_padding_efficiency": emitted / (plan.batch * plan.windows * plan.step),
           "equal_padding_efficiency": base_frames / (args.clips * ragged_eq.windows * plan.step)}
    for k, ts in times.items():
        med = float(np.median(ts))
        res[k] = {"median_s": med, "min_s": float(np.min(ts)), "max_s": float(np.max(ts)), "frames_per_s": frames[k] / med}
    res["a_over_b"] = res["a_ragged_mix"]["frames_per_s"] / res["b_one_by_one_mix"]["frames_per_s"]
    res["c_ragged_over_captured_time"] = res["c_ragged_equal"]["median_s"] / res["c_captured_equal"]["median_s"]
    res["c_replay_ragged_over_captured_time"] = res["c_ragged_replay"]["median_s"] / res["c_captured_replay"]["median_s"]
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
