"""Caller plumbing of the hot path: the timed span of the reference demo
(/root/reference/test_emage_audio.py:16-47, twin train_emage_audio.py:33-102) without audio file
decoding and npz writing: inference() -> indices from the concatenated logits -> full-length
decode(get_global_motion=True)."""
from __future__ import annotations

import torch

from . import _lib, ops
from .emage_audio import engine as _E
from .emage_audio.engine import PARTS, select_inputs

_OVERFLOW = ("fp16x3: a GEMM operand exceeded the fp16 range (|x| > 1023 after the x64 pre-scale) and the result is NaN - "
             "use engine.set_precision('bf16x6') for this checkpoint (model.inference() outside a captured graph retries "
             "in bf16x6 by itself)")


@torch.no_grad()
def generate(model, motion_vq, audio, speaker_id=None, masked_motion=None, mask=None, ref_trans=None):
    """audio (bs, n) float32 16 kHz.  Returns (latent_dict, pred_dict) like T.py:32 and T.py:44-47."""
    dev = next(model.parameters()).device
    bs = audio.shape[0]
    if speaker_id is None:
        speaker_id = torch.zeros(bs, 1, dtype=torch.long, device=dev)                  # T.py:19
    lat = model.inference(audio, speaker_id, motion_vq, masked_motion=masked_motion, mask=mask)
    # fp16 operand planes turn an out-of-range activation into inf - inf = NaN in the consuming GEMM; a NaN anywhere
    # upstream reaches the logits (cls_* = MLP(rec_*)), which the argmax kernels read anyway: they raise the flag.
    generate.nonfinite = ops.zero_flag(dev) if ops.plane_format() == "fp16" else None
    cfg = model.cfg.to_dict()
    idx = {p: ops.row_argmax(lat["cls_" + p], nonfinite=generate.nonfinite) for p in PARTS}       # T.py:39-42
    if generate.nonfinite is not None:
        capturing = lat["rec_face"].is_cuda and torch.cuda.is_current_stream_capturing()
        if not capturing and bool(generate.nonfinite):
            raise _lib.PmError(_OVERFLOW)
    index, latent = select_inputs(cfg, lat, idx)
    if ref_trans is None:
        ref_trans = torch.zeros(1, 3, device=dev)                                       # trans[:,0], T.py:30,47
    pred = motion_vq.decode(
        face_latent=latent["face"], upper_latent=latent["upper"], lower_latent=latent["lower"],
        hands_latent=latent["hands"], face_index=index["face"], upper_index=index["upper"],
        lower_index=index["lower"], hands_index=index["hands"], get_global_motion=True, ref_trans=ref_trans)
    return lat, pred


generate.nonfinite = None


class CapturedPipeline:
    """generate() captured once into a CUDA graph for a fixed (batch, n_samples) and replayed per call.

    The hot path is ~10^3 small kernel launches per step; replaying them as one graph removes the Python /
    launch latency between kernels (B200 guide: capture launch-bound inner loops in CUDA graphs).  Inputs
    are copied into static device buffers, outputs are static tensors owned by this object (valid until
    the next call).  Only the default-input form of the demo (masked_motion=None, mask=None) is captured.
    """

    def __init__(self, model, motion_vq, batch: int, n_samples: int, warmup: int = 2, body_priority: bool = True):
        self.model, self.vq = model, motion_vq
        dev = next(model.parameters()).device
        self.device = dev
        self.audio = torch.zeros(batch, n_samples, device=dev)
        self.speaker_id = torch.zeros(batch, 1, dtype=torch.long, device=dev)
        self.ref_trans = torch.zeros(1, 3, device=dev)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):                        # warm-up off the capture: lazy packing, attributes
            for _ in range(warmup):
                generate(model, motion_vq, self.audio, self.speaker_id, ref_trans=self.ref_trans)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        before = ops.launch_count
        # The capture stream carries the longest dependency chain (the body stack: 1 + 8 layers per window); the face /
        # refine / part branches fork onto default-priority side streams.  Capturing on a high-priority stream makes the
        # kernel nodes of the critical chain win when both have thread blocks ready (a 96-CTA GEMM leaves 52 SMs free,
        # which the other branch's blocks share): measured effect in profiles/README.md.
        self.capture_stream = torch.cuda.Stream(device=dev, priority=-1) if body_priority else None
        with torch.cuda.graph(self.graph, stream=self.capture_stream):
            self.latent, self.pred = generate(model, motion_vq, self.audio, self.speaker_id, ref_trans=self.ref_trans)
        self.kernels_per_replay = ops.launch_count - before
        self.nonfinite = generate.nonfinite                  # fp16 planes only: in-graph overflow flag (else None)

    @torch.no_grad()
    def __call__(self, audio, speaker_id=None):
        """audio: (batch, n_samples) float32, host (pinned for async copies) or device."""
        self.audio.copy_(audio, non_blocking=True)
        if speaker_id is not None:
            self.speaker_id.copy_(speaker_id, non_blocking=True)
        self.graph.replay()
        ops.launch_count += self.kernels_per_replay
        if self.nonfinite is not None and bool(self.nonfinite):     # one 4-byte read back per step (fp16 planes only)
            raise _lib.PmError(_OVERFLOW)
        return self.latent, self.pred


def _ragged_decode(model, motion_vq, lat, limits, ref_trans, dev):
    """generate()'s tail for a ragged batch: indices from the concatenated logits and the full-length decode over the
    capacity frames, every conv limited to each clip's out_len.  Returns (pred dict, nonfinite flag or None)."""
    flag = ops.zero_flag(dev) if ops.plane_format() == "fp16" else None
    idx = {p: ops.row_argmax(lat["cls_" + p], nonfinite=flag) for p in PARTS}                     # T.py:39-42
    index, latent = select_inputs(model.cfg.to_dict(), lat, idx)
    if ref_trans is None:
        ref_trans = torch.zeros(1, 3, device=dev)
    pred = motion_vq.engine().decode(index, latent, get_global_motion=True, ref_trans=ref_trans, row_limit=limits.out_len)
    return pred, flag


def _split_clips(lat, pred, out_len):
    """Per-clip views (batch dim 1, out_len frames) of capacity-shaped outputs."""
    return [({k: v[b:b + 1, :n] for k, v in lat.items()}, {k: v[b:b + 1, :n] for k, v in pred.items()})
            for b, n in enumerate(out_len)]


def _ragged_inputs(audios, batch, max_samples, dev):
    if len(audios) == 0 or len(audios) > batch:
        raise ValueError(f"a ragged batch holds 1 to {batch} clips, got {len(audios)}")
    lens = [int(a.shape[-1]) for a in audios]
    if max(lens) > max_samples:
        raise ValueError(f"clip of {max(lens)} samples exceeds the capacity of {max_samples}")
    return lens


@torch.no_grad()
def generate_ragged(model, motion_vq, audios, speaker_ids=None, ref_trans=None, masked_motion=None, mask=None):
    """generate() for a list of clips of different lengths, run as ONE batched schedule (engine.RaggedPlan).
    audios: list of (n_i,) or (1, n_i) float32 16 kHz tensors; speaker_ids: optional list of ints / (1,1) tensors.
    Returns, per clip, the (latent_dict, pred_dict) generate(model, motion_vq, audio_i[None], speaker_id_i) returns
    (batch dim 1, the clip's own frame count).  Per-clip masked motion is not supported."""
    if masked_motion is not None or mask is not None:
        raise ValueError("generate_ragged runs the default (unmasked) form only: pass masked_motion / mask to generate()")
    dev = next(model.parameters()).device
    audios = [a.reshape(-1) for a in audios]
    cfg = model.cfg.to_dict()
    plan = _E.RaggedPlan([a.shape[0] for a in audios], int(cfg["pose_length"]), int(cfg["seed_frames"]))
    audio = torch.zeros(plan.batch, plan.capacity_samples, device=dev)
    for b, a in enumerate(audios):                     # samples beyond the capacity belong to no window
        m = min(a.shape[0], plan.capacity_samples)
        audio[b, :m] = a[:m].to(device=dev, dtype=torch.float32)
    spk = torch.zeros(plan.batch, 1, dtype=torch.long, device=dev)
    if speaker_ids is not None:
        for b, sid in enumerate(speaker_ids):
            spk[b, 0] = int(sid)
    limits = _E.RaggedLimits(plan, dev)
    eng, vq = model._eng(), motion_vq.engine()
    lat = _E.guarded(lambda: _E.run_inference_ragged(eng, vq, audio, limits, spk), lambda out: [out["cls_" + p] for p in PARTS])
    pred, flag = _ragged_decode(model, motion_vq, lat, limits, ref_trans, dev)
    if flag is not None and bool(flag):
        raise _lib.PmError(_OVERFLOW)
    return _split_clips(lat, pred, [int(n) for n in plan.out_len[:plan.n_clips]])


class RaggedPipeline:
    """generate_ragged() captured once into a CUDA graph at a fixed capacity - `batch` clips of up to `max_samples`
    samples - and replayed for any list of clips within it.  A call copies the audio into a static zero-padded buffer
    and the batch's plan tables into a static device buffer (one small copy), replays the graph and returns
    per-clip views of static outputs, valid until the next call.  Clip slots a call does not use have no windows."""

    def __init__(self, model, motion_vq, batch: int, max_samples: int, warmup: int = 2, body_priority: bool = True):
        self.model, self.vq = model, motion_vq
        dev = next(model.parameters()).device
        self.device, self.batch, self.max_samples = dev, int(batch), int(max_samples)
        cfg = model.cfg.to_dict()
        self.window, self.pre = int(cfg["pose_length"]), int(cfg["seed_frames"])
        full = _E.RaggedPlan([self.max_samples] * self.batch, self.window, self.pre)
        self.windows = full.windows
        self.audio = torch.zeros(self.batch, full.capacity_samples, device=dev)
        self.speaker_id = torch.zeros(self.batch, 1, dtype=torch.long, device=dev)
        self.ref_trans = torch.zeros(1, 3, device=dev)
        self.limits = _E.RaggedLimits(full, dev)
        eng, vq = model._eng(), motion_vq.engine()

        def step():
            lat = _E.run_inference_ragged(eng, vq, self.audio, self.limits, self.speaker_id)
            pred, flag = _ragged_decode(model, motion_vq, lat, self.limits, self.ref_trans, dev)
            return lat, pred, flag

        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):                        # warm-up off the capture: lazy packing, attributes
            for _ in range(warmup):
                step()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        before = ops.launch_count
        self.capture_stream = torch.cuda.Stream(device=dev, priority=-1) if body_priority else None
        with torch.cuda.graph(self.graph, stream=self.capture_stream):
            self.latent, self.pred, self.nonfinite = step()
        self.kernels_per_replay = ops.launch_count - before

    def plan(self, n_samples):
        return _E.RaggedPlan(n_samples, self.window, self.pre, batch=self.batch, windows=self.windows)

    @torch.no_grad()
    def load(self, audios, speaker_ids=None):
        """Stage a batch without running it: audio into the static zero-padded buffer (samples beyond the capacity
        belong to no window), speaker ids and the plan tables (one host -> device copy).  Returns the plan."""
        audios = [a.reshape(-1) for a in audios]
        _ragged_inputs(audios, self.batch, self.max_samples, self.device)
        plan = self.plan([a.shape[0] for a in audios])
        cap = self.audio.shape[1]
        for b in range(self.batch):
            m = min(audios[b].shape[0], cap) if b < len(audios) else 0
            if m:
                self.audio[b, :m].copy_(audios[b][:m], non_blocking=True)
            if m < cap:
                self.audio[b, m:].zero_()
        spk = torch.zeros(self.batch, 1, dtype=torch.long)
        if speaker_ids is not None:
            for b, sid in enumerate(speaker_ids):
                spk[b, 0] = int(sid)
        self.speaker_id.copy_(spk)
        self.limits.load(plan)
        return plan

    def replay(self):
        """Run the captured step on whatever load() staged last."""
        self.graph.replay()
        ops.launch_count += self.kernels_per_replay

    @torch.no_grad()
    def __call__(self, audios, speaker_ids=None):
        """audios: list of up to `batch` (n_i,) / (1, n_i) float32 tensors, n_i <= max_samples."""
        plan = self.load(audios, speaker_ids)
        self.replay()
        if self.nonfinite is not None and bool(self.nonfinite):     # one 4-byte read back per step (fp16 planes only)
            raise _lib.PmError(_OVERFLOW)
        return _split_clips(self.latent, self.pred, [int(n) for n in plan.out_len[:plan.n_clips]])
