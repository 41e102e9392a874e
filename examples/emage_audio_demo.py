#!/usr/bin/env python
"""Audio folder -> BEAT-format motion npz files: the reference demo (test_emage_audio.py:71-105) on the B200 path.

    python examples/emage_audio_demo.py --checkpoint /path/to/emage_audio --audio_folder ./wavs --save_folder ./out
    python examples/emage_audio_demo.py --synthetic --audio_folder ./wavs            # seeded random weights (no network)
    python examples/emage_audio_demo.py --checkpoint DIR --audio_folder ./wavs --batch 16   # ragged batches of 16 files

`--checkpoint` is a local copy of the Hugging Face repo layout the reference downloads (config.json +
model.safetensors at the top level, VQ models under emage_vq/{face,upper,lower,hands,global}).
"""
import argparse
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from models.emage_audio import EmageAudioModel, EmageVAEConv, EmageVQModel, EmageVQVAEConv  # noqa: E402  (B200 drop-in)
from pantomatrix_b200.audio_io import load_audio  # noqa: E402
from pantomatrix_b200.motion_io import beat_format_save  # noqa: E402
from pantomatrix_b200.pipeline import generate, generate_ragged  # noqa: E402


def load_models(args, device):
    if args.synthetic:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from synthetic_models import build_product
        return build_product(seed=0, device=device)
    ck = args.checkpoint
    vq = {p: EmageVQVAEConv.from_pretrained(ck, subfolder=f"emage_vq/{p}").to(device) for p in ("face", "upper", "lower", "hands")}
    glob = EmageVAEConv.from_pretrained(ck, subfolder="emage_vq/global").to(device)
    motion_vq = EmageVQModel(face_model=vq["face"], upper_model=vq["upper"], lower_model=vq["lower"],
                             hands_model=vq["hands"], global_model=glob).to(device).eval()
    return EmageAudioModel.from_pretrained(ck).to(device).eval(), motion_vq


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--audio_folder", default="./examples/audio")
    ap.add_argument("--save_folder", default="./examples/motion")
    ap.add_argument("--checkpoint", default=None)
    ap.add_argument("--synthetic", action="store_true")
    ap.add_argument("--batch", type=int, default=1,
                    help="files per ragged batch (sorted by length, run as one batched schedule); 1: one file at a time")
    args = ap.parse_args()
    if args.batch < 1:
        ap.error("--batch must be >= 1")
    if not args.synthetic and not args.checkpoint:
        ap.error("give --checkpoint DIR or --synthetic")
    os.makedirs(args.save_folder, exist_ok=True)
    device = torch.device("cuda")                      # no CPU fallback by design
    model, motion_vq = load_models(args, device)
    sr, fps = model.cfg.audio_sr, model.cfg.pose_fps
    files = sorted(f for f in os.listdir(args.audio_folder) if f.endswith(".wav"))
    frames, t0 = 0, time.time()
    audios = {name: torch.from_numpy(load_audio(os.path.join(args.audio_folder, name), sr=sr)) for name in files}
    if args.batch == 1:
        results = ((name, generate(model, motion_vq, audios[name].unsqueeze(0).to(device))[1]) for name in files)
    else:                                              # similar lengths together: less padding per ragged batch
        order = sorted(files, key=lambda f: audios[f].shape[0])
        groups = [order[i:i + args.batch] for i in range(0, len(order), args.batch)]
        results = ((name, pred) for g in groups
                   for name, (_, pred) in zip(g, generate_ragged(model, motion_vq, [audios[f].to(device) for f in g])))
    for name, pred in results:
        t = pred["motion_axis_angle"].shape[1]
        beat_format_save(os.path.join(args.save_folder, os.path.splitext(name)[0] + "_output.npz"),
                         pred["motion_axis_angle"].cpu().numpy().reshape(t, -1), upsample=30 // fps,
                         expressions=pred["expression"].cpu().numpy().reshape(t, -1),
                         trans=pred["trans"].cpu().numpy().reshape(t, -1))
        frames += t
    print(f"generate total {frames / fps:.2f} seconds motion in {time.time() - t0:.2f} seconds")


if __name__ == "__main__":
    main()
