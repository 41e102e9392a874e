"""Execution engine of the EMAGE hot path: packed device weights + the kernel schedule.

Host logic only (Python, like the reference); every arithmetic op is a libpm_emage.so kernel reached
through pantomatrix_b200.ops.  Citations: M.py = /root/reference/models/emage_audio/modeling_emage_audio.py,
P.py = .../processing_emage_audio.py.

Schedule differences from the reference that do not change results beyond fp32 rounding:
  * BatchNorm (eval) is folded into the preceding conv at pack time (P.py:285-291).
  * Everything that depends only on audio is hoisted out of the sequential window loop and batched over
    all windows of all clips: both WavEncoders, audio_body_motion_proj, the audio half of
    audio_face_motion_proj and the cross-attention K/V projections of the 8 audio_motion_cross_attn
    layers (SURVEY.md section 3.3).  Each window still sees its own zero-padded audio slice, as in the
    reference (M.py:393-396), so window-local conv results are reproduced exactly.
  * In-loop VQ decodes only produce the seed frames (M.py:418): the conv decoders are run on the last
    seed_frames + (5 + vae_layer) frames of the window, which covers their receptive field (seed_decode_frames()).
  * Window outputs are written by their final GEMMs straight into the accumulated result tensors, and the tail frames
    the seed decode needs are read from there as strided views: the steady-state step contains no torch kernels.
"""
from __future__ import annotations

import numpy as np
import torch

from .. import _lib, ops

PARTS = ("face", "upper", "hands", "lower")
# WavEncoder geometry P.py:300-307: (stride, first-conv padding, has downsample branch)
WAV_BLOCKS = ((5, 1600, True), (6, 0, True), (1, 7, False), (6, 0, True), (1, 7, False), (3, 0, True))
NHEAD = 4


def _taps(w: torch.Tensor) -> torch.Tensor:
    """conv weight (cout, cin, k) -> tap-major (k, cout, cin)."""
    return w.permute(2, 0, 1).contiguous()


def _fold_bn(sd, conv, bn, eps=1e-5):
    w, b = sd[conv + ".weight"].double(), sd[conv + ".bias"].double()
    s = sd[bn + ".weight"].double() / torch.sqrt(sd[bn + ".running_var"].double() + eps)
    return (w * s[:, None, None]).float(), ((b - sd[bn + ".running_mean"].double()) * s + sd[bn + ".bias"].double()).float()


def wav_block_lens(n: int) -> list[int]:
    """Rows each WavEncoder block emits for n samples (P.py:300-307 conv arithmetic); a block's k=15 / pad 7 second
    conv keeps the row count of its first."""
    lens, length = [], n
    for stride, pad, _ in WAV_BLOCKS:
        length = (length + 2 * pad - 15) // stride + 1
        lens.append(length)
    return lens


def wav_out_len(n: int) -> int:
    """Frames a WavEncoder emits for n samples (P.py:300-307 conv arithmetic)."""
    return wav_block_lens(n)[-1]


# Arithmetic engine of every Conv1d / Linear ("tap-GEMM"): 0 = fp32 SIMT kernel, 1/2/3 = tcgen05 tensor cores with
# 1 / 2 / 3 operand planes (csrc/pm_tapgemm_tc.cu).
#   fp16x3 (default)  two IEEE fp16 planes (22 mantissa bits), 3 tensor-core products per fp32 product.  Measured on
#                     B200 (round 2, profiles/README.md): all 38 400 codes of the BASELINE batch identical to the fp32
#                     reference, latent error 4.3e-4 (bf16x6: 3.8e-4), 24 ms per step against 31 ms.  Operands must stay
#                     below 65504 / 64 (activations are pre-scaled by 64, ops.F16_ACT_SCALE): pipeline.py checks the
#                     outputs for the NaN an overflow would leave and names bf16x6 as the way out.
#   bf16x6            three bf16 planes, 6 products: same accuracy, no range limit (fp32 exponent range), 1.3x slower.
#   bf16x3 / bf16     faster, below the parity gates (measured agreement in profiles/README.md).
#   fp32              exact-order fp32 SIMT engine (reference engine of the tests).
PRECISIONS = {"fp32": 0, "bf16": 1, "bf16x3": 2, "bf16x6": 3, "fp16x3": 2}
PLANE_FORMAT = {"fp16x3": "fp16"}
DEFAULT_PRECISION = __import__("os").environ.get("PM_EMAGE_PRECISION", "fp16x3")     # PM_EMAGE_PRECISION overrides
_STATE = {"nsplit": PRECISIONS[DEFAULT_PRECISION], "fork": True,   # fork: overlap independent branches on side streams
          "precision": DEFAULT_PRECISION,
          # clip-group lanes of the window loop (run_inference).  Measured at batch 32: 1 lane 19.91 ms, 2 lanes 19.59,
          # 4 lanes 19.49 per step - a 2 % gain for 2-4x the kernel launches, so one lane is the default.
          "groups": int(__import__("os").environ.get("PM_EMAGE_GROUPS", "1"))}
ops.set_plane_format(PLANE_FORMAT.get(DEFAULT_PRECISION, "bf16"))


def set_precision(name: str) -> None:
    if name not in PRECISIONS:
        raise ValueError(f"precision must be one of {sorted(PRECISIONS)}")
    _STATE["nsplit"] = PRECISIONS[name]
    _STATE["precision"] = name
    ops.set_plane_format(PLANE_FORMAT.get(name, "bf16"))


def get_precision() -> str:
    name = _STATE.get("precision")
    if name in PRECISIONS and PRECISIONS[name] == _STATE["nsplit"]:
        return name
    return next(k for k, v in PRECISIONS.items() if v == _STATE["nsplit"])     # _STATE["nsplit"] was set directly (tests)


def _pk(nsplit: int) -> int:
    """Cache key of packed weights: split count + plane format."""
    return nsplit | (ops.FMT_F16 if ops.plane_format() == "fp16" else 0)


def guarded(run, checked):
    """Run `run()` in the current precision; in the fp16x3 engine verify afterwards that no GEMM operand left the
    fp16 range and, if one did, recompute in bf16x6 (same accuracy, fp32 exponent range) - still on the GPU, with a
    warning.  `checked(result)` returns the fp32 tensors whose NaN would reveal the overflow (an out-of-range operand
    becomes inf - inf = NaN in the consuming GEMM and propagates to every output).  Inside a CUDA-graph capture nothing
    can be read back: the captured pipeline carries the flag itself (pipeline.CapturedPipeline)."""
    out = run()
    if ops.plane_format() != "fp16":
        return out
    tensors = [t for t in checked(out) if t is not None]
    if not tensors or not tensors[0].is_cuda or torch.cuda.is_current_stream_capturing():
        return out
    flag = ops.zero_flag(tensors[0].device)
    for t in tensors:
        ops.row_argmax(t, nonfinite=flag)                # the kernel that reads the logits anyway; indices discarded
    if not bool(flag):
        return out
    import warnings
    warnings.warn("fp16x3: a GEMM operand exceeded the fp16 range (|x| > 1023 after the x64 pre-scale); "
                  "recomputing this call with engine.set_precision('bf16x6') - select it up front for this checkpoint")
    prev = get_precision()
    set_precision("bf16x6")
    try:
        return run()
    finally:
        set_precision(prev)


def _record_stream(obj, stream):
    if isinstance(obj, torch.Tensor):
        if obj.is_cuda:
            obj.record_stream(stream)
    elif isinstance(obj, dict):
        for v in obj.values():
            _record_stream(v, stream)
    elif isinstance(obj, (list, tuple)):
        for v in obj:
            _record_stream(v, stream)


class _Fork:
    """Run independent branches of the schedule on side CUDA streams and join them on the current stream
    (the face decoder || the body stack, the three refine decoders, the four VQ part decoders).  The M = 2048
    GEMMs of one branch fill only ~100 of the 148 SMs; overlapping branches fills the rest.  Works inside
    CUDA-graph capture (event waits become graph edges).  Sequential when there is no CUDA device (tests)."""

    def __init__(self, n_side):
        self.n_side, self.streams = n_side, None

    def run(self, fns):
        if not torch.cuda.is_available() or len(fns) == 1 or not _STATE["fork"]:
            return [fn() for fn in fns]
        if self.streams is None:
            self.streams = [torch.cuda.Stream() for _ in range(self.n_side)]
        cur = torch.cuda.current_stream()
        ready = torch.cuda.Event()
        ready.record(cur)
        results = [None] * len(fns)
        for i in range(1, len(fns)):
            st = self.streams[i - 1]
            st.wait_event(ready)
            with torch.cuda.stream(st):
                results[i] = fns[i]()
        results[0] = fns[0]()
        for i in range(1, len(fns)):
            cur.wait_stream(self.streams[i - 1])
            _record_stream(results[i], cur)
        return results


class _Conv:
    """One Conv1d / Linear: fp32 tap-major weights (taps, cout, cin) + lazily packed bf16 planes."""
    __slots__ = ("w", "b", "stride", "pad", "_packed", "_next")

    def __init__(self, w, b, stride=1, pad=0):
        self.w, self.b, self.stride, self.pad = w, b, stride, pad
        self._packed = {}
        self._next = None          # the GEMM that followed this one last time (learned; see _prefetch_hint)

    def _prefetch_hint(self, ns):
        """Weights are read once per window and do not fit L2, so each GEMM prefetches the NEXT GEMM's packed
        weights into L2 while it runs.  The schedule is static, so "next" is simply whichever GEMM was issued
        after this one on the previous pass (a wrong guess only costs a useless prefetch)."""
        prev = _STATE.get("prev_conv")
        if prev is not None and prev is not self:
            prev._next = self
        _STATE["prev_conv"] = self
        nxt = self._next
        return nxt._packed[_pk(ns)].t if (nxt is not None and _pk(ns) in nxt._packed) else None

    def packed(self, nsplit):
        """bf16 planes for the tensor-core engine.  A stride-s conv is packed as the equivalent stride-1 conv
        over the (rows/s, s*cin) view of its input: tap k = s*q + r lands in tap q, channel block r; taps
        beyond the kernel size are zero."""
        key = _pk(nsplit)
        if key not in self._packed:
            w, s = self.w, self.stride
            if s > 1:
                taps, cout, cin = w.shape
                wp = torch.zeros(-(-taps // s), cout, s * cin, device=w.device, dtype=w.dtype)
                for k in range(taps):
                    wp[k // s, :, (k % s) * cin:(k % s + 1) * cin] = w[k]
                w = wp
            self._packed[key] = ops.PackedW(w, nsplit)
        return self._packed[key]

    def __call__(self, x, act=ops.ACT_NONE, slope=0.0, residual=None, out=None, want="f", out_slack=0, row_limit=None):
        """x: fp32 tensor, ops.Planes or ops.Act.  want: "f" (fp32 tensor returned), "p" (bf16 planes only) or
        "fp" (both); with planes requested an ops.Act is returned.  In fp32 mode planes do not exist: the fp32
        tensor is always produced and returned (wrapped in an Act when planes were asked for).
        row_limit: per-clip valid output rows of a ragged batch (int32 device tensor, None = all rows)."""
        ns = _STATE["nsplit"]
        residual = _f32(residual)
        lim = {} if row_limit is None else {"row_limit": row_limit}          # no limit: exactly the plain call
        if ns == 0:
            y = ops.tapgemm(_f32(x), self.w, self.b, stride=self.stride, pad=self.pad, act=act, slope=slope,
                            residual=residual, out=out, **lim)
            return y if want == "f" else ops.Act(y, None)
        taps, cout, _ = self.w.shape
        s = self.stride
        want_f, out_ns = "f" in want, (ns if "p" in want else 0)
        pf = self._prefetch_hint(ns)
        if s == 1:
            a = _planes(x, ns)
            batch, rows = a.batch, a.rows
            rows_out = rows + 2 * self.pad - taps + 1
            flat = (taps == 1 and batch > 1 and a.t.stride(1) == rows * a.t.stride(2)
                    and (out is None or out.is_contiguous()) and (residual is None or residual.is_contiguous()))
            if want_f and out is None:
                out = torch.empty(batch, rows_out, cout, device=a.t.device, dtype=torch.float32)
            if flat:                                       # a Linear over all clips is one tall matrix
                _, pl = ops.tapgemm_tc(a.flat(), self.packed(ns), self.b, rows_out=batch * rows, act=act, slope=slope,
                                       want_f32=want_f, out=None if out is None else out.view(1, batch * rows, cout),
                                       residual=None if residual is None else residual.view(1, batch * rows, cout),
                                       out_nsplit=out_ns, out_slack=out_slack, prefetch=pf,
                                       **({} if row_limit is None else {"row_limit": row_limit, "rows_per_clip": rows}))
                if pl is not None:                         # back to the (clips, rows) view
                    pl = ops.Planes(pl.t.view(pl.t.shape[0], batch, rows, pl.t.shape[3]), rows, cout, pl.slack)
            else:
                _, pl = ops.tapgemm_tc(a, self.packed(ns), self.b, rows_out=rows_out, pad=self.pad, act=act, slope=slope,
                                       residual=residual, want_f32=want_f, out=out, out_nsplit=out_ns, out_slack=out_slack,
                                       prefetch=pf, **lim)
            return out if want == "f" else ops.Act(out, pl)
        assert self.pad == 0
        a = _planes(x, ns, need_slack=s)
        batch, rows, cin = a.batch, a.rows, a.ch
        assert a.t.stride(2) == cin and a.t.stride(1) == rows * cin, "strided view needs dense (clips*rows, C) planes"
        rows_out = (rows - taps) // s + 1
        o, pl = ops.tapgemm_tc(a, self.packed(ns), self.b, rows_out=rows_out, act=act, slope=slope, residual=residual,
                               want_f32=want_f, out=out, out_nsplit=out_ns, out_slack=out_slack, prefetch=pf,
                               a_view=(-(-rows // s), s * cin, s * cin), **lim)
        return o if want == "f" else ops.Act(o, pl)


def _f32(x):
    """The fp32 tensor of an activation (Act or plain tensor)."""
    if isinstance(x, ops.Act):
        assert x.f is not None, "this consumer needs the fp32 copy"
        return x.f
    return x


def _planes(x, ns, need_slack=0):
    """bf16 planes of an activation: reuse the producer's planes when present (and padded enough), else convert."""
    if isinstance(x, ops.Planes):
        assert x.slack >= need_slack
        return x
    if isinstance(x, ops.Act):
        if x.p is not None and x.p.nsplit == ns and x.p.slack >= need_slack and x.p.t.dtype == ops._PLANE_DTYPE:
            return x.p
        x = x.f
    return ops.split_bf16(x, ns, slack_rows=need_slack)


def _ns():
    return _STATE["nsplit"]


class _Linear(_Conv):
    def __init__(self, sd, prefix=None, w=None, b=None):
        if prefix is not None:
            w, b = sd[prefix + ".weight"], sd[prefix + ".bias"]
        super().__init__(w.contiguous().unsqueeze(0), None if b is None else b.contiguous())


class _MLP:
    """P.py:316-326."""

    def __init__(self, sd, p):
        self.fc1, self.fc2 = _Linear(sd, p + ".fc1"), _Linear(sd, p + ".fc2")

    def __call__(self, x, out=None, want="f", row_limit=None):
        return self.fc2(self.fc1(x, act=ops.ACT_LEAKY, slope=0.1, want="p", row_limit=row_limit), out=out, want=want,
                        row_limit=row_limit)


class _ConvStack:
    """k=3 conv stacks: VQEncoderV5/V6 (P.py:189-235) and VQDecoderV5 (P.py:237-261)."""

    def __init__(self, sd, prefix, kind, n_layer):
        c = lambda i, sub="": _Conv(_taps(sd[f"{prefix}.main.{i}{sub}.weight"]), sd[f"{prefix}.main.{i}{sub}.bias"].contiguous(), 1, 1)
        self.steps = []           # ("conv", conv, act) | ("res", conv_a, conv_b)
        if kind == "encoder":
            for i in range(n_layer):
                self.steps.append(("conv", c(3 * i), True))
                self.steps.append(("res", c(3 * i + 2, ".model.0"), c(3 * i + 2, ".model.2")))
        else:
            self.steps.append(("res", c(0, ".model.0"), c(0, ".model.2")))
            self.steps.append(("res", c(1, ".model.0"), c(1, ".model.2")))
            for i in range(n_layer):
                self.steps.append(("conv", c(2 + 2 * i), True))
            self.steps.append(("conv", c(2 + 2 * n_layer), False))

    def __call__(self, x, want="f", row_limit=None):
        """x: tensor / Act (a ResBlock needs its fp32 copy for the skip).  Intermediate activations travel as
        fp32 + bf16 planes; only the last step honours `want`.  row_limit: per-clip valid rows of a ragged batch -
        every conv zeroes the rows beyond, which is the zero padding the next conv of the clip alone would read."""
        last = len(self.steps) - 1
        rl = row_limit
        for i, step in enumerate(self.steps):
            w = want if i == last else "fp"
            if step[0] == "conv":
                x = step[1](x, act=ops.ACT_LEAKY if step[2] else ops.ACT_NONE, slope=0.2, want=w, row_limit=rl)
            else:
                x = step[2](step[1](x, act=ops.ACT_LEAKY, slope=0.2, want="p", row_limit=rl), residual=x, want=w, row_limit=rl)
        return x


class _WavEncoder:
    """P.py:263-314 with BatchNorm folded; input is a set of (clip, window) waveform slices."""

    def __init__(self, sd, p, blocks=WAV_BLOCKS):
        self.blocks = []
        for i, (stride, pad, has_ds) in enumerate(blocks):
            q = f"{p}.feat_extractor.{i}"
            w1, b1 = _fold_bn(sd, q + ".conv1", q + ".bn1")
            w2, b2 = _fold_bn(sd, q + ".conv2", q + ".bn2")
            ds = _fold_bn(sd, q + ".downsample.0", q + ".downsample.1") if has_ds else None
            if i == 0:
                self.stem = (w1.reshape(w1.shape[0], -1).contiguous(), b1.contiguous(),
                             ds[0].reshape(ds[0].shape[0], -1).contiguous(), ds[1].contiguous(), stride, pad)
                self.blocks.append((None, _Conv(_taps(w2), b2.contiguous(), 1, 7), None))
            else:
                self.blocks.append((_Conv(_taps(w1), b1.contiguous(), stride, pad), _Conv(_taps(w2), b2.contiguous(), 1, 7),
                                    _Conv(_taps(ds[0]), ds[1].contiguous(), stride, pad) if ds else None))

    def __call__(self, audio, offset, a_ws, windows, n_samples, limits=None):
        """audio (bs, n) contiguous; returns (windows*bs, frames, out_dim), window-major.
        limits: ragged batch - (samples per slice, [valid rows after each block]), int32 device tensors over the
        window-major slices (RaggedPlan); None: every slice is n_samples long."""
        bs, n = audio.shape
        w1, b1, wd, bd, stride, pad = self.stem
        n_valid, rows = limits if limits is not None else (None, [None] * len(self.blocks))
        y, sc = ops.wav_stem(audio, n, a_ws, bs, windows, n_samples, w1, b1, wd, bd, stride=stride, pad=pad,
                             slope=0.01, offset=offset, nsplit=_ns(), **({} if n_valid is None else {"n_valid": n_valid}))
        # A block's output feeds the next block's convs as (possibly strided) GEMM operand - planes - and, only where
        # that block has no downsample conv, as its identity shortcut - fp32.  (The first block's output is 0.25 GB
        # per encoder in fp32 at the BASELINE batch: not writing it is the point.)
        last = len(self.blocks) - 1
        form = lambda i: "f" if i == last else ("p" if self.blocks[i + 1][2] is not None else "fp")
        x = self.blocks[0][1](y, act=ops.ACT_LEAKY, slope=0.01, residual=sc, want=form(0), out_slack=8, row_limit=rows[0])
        for i, (conv1, conv2, ds) in enumerate(self.blocks[1:], 1):
            y = conv1(x, act=ops.ACT_LEAKY, slope=0.01, want="p", row_limit=rows[i])
            sc = ds(x) if ds is not None else x          # only read as conv2's residual, on rows conv2 computes
            x = conv2(y, act=ops.ACT_LEAKY, slope=0.01, residual=sc, want=form(i), out_slack=8, row_limit=rows[i])
        return x


class _Attn:
    """nn.MultiheadAttention weights (packed in_proj (3E,E): Q | K | V rows)."""

    def __init__(self, sd, p, E):
        w, b = sd[p + ".in_proj_weight"], sd[p + ".in_proj_bias"]
        self.qkv = _Linear(None, w=w, b=b)
        self.q = _Linear(None, w=w[:E], b=b[:E])
        self.kv = _Linear(None, w=w[E:], b=b[E:])
        self.out = _Linear(sd, p + ".out_proj")
        self.E = E


class _Layer:
    """Post-norm nn.TransformerEncoderLayer / DecoderLayer (ReLU FFN), M.py:238-250."""

    def __init__(self, sd, p, E, cross):
        self.E = E
        self.sa = _Attn(sd, p + ".self_attn", E)
        self.ca = _Attn(sd, p + ".multihead_attn", E) if cross else None
        self.l1, self.l2 = _Linear(sd, p + ".linear1"), _Linear(sd, p + ".linear2")
        n = 3 if cross else 2
        self.norms = [(sd[f"{p}.norm{i + 1}.weight"].contiguous(), sd[f"{p}.norm{i + 1}.bias"].contiguous()) for i in range(n)]

    def project_memory(self, mem):
        """K|V projection of a cross-attention memory (bs, tk, E) -> (bs, tk, 2E): fp32, or the fp16 operand planes
        the tensor-core attention kernel reads in place."""
        return self.ca.kv(mem, want="p" if _attn_tc() else "f")

    def __call__(self, x, mem_kv=None, want="f", q_len=None, k_len=None):
        """x: fp32 tensor or Act(f, p) of (bs, t, E).  Returns the layer output in the requested form.
        Ragged batch: q_len = per-clip valid rows of x (the self-attention keys too), k_len = per-clip memory keys."""
        sa = {} if q_len is None else {"q_len": q_len, "k_len": q_len}
        ca = {} if q_len is None else {"q_len": q_len, "k_len": k_len}
        ns = _ns()
        xf = _f32(x)
        bs, t, E = xf.shape
        hd = E // NHEAD
        tc = _attn_tc()
        if tc:                                  # packed q|k|v planes straight from the GEMM epilogue, read in place by TMA
            qkv = self.sa.qkv(x, want="p").p
            att = ops.attention_tc(qkv, 0, qkv, E, qkv, 2 * E, bs, NHEAD, t, t, hd, nsplit=ns, **sa)
        else:
            qkv = self.sa.qkv(x).view(bs * t, 3 * E)
            att = ops.attention(qkv[:, :E], qkv[:, E:2 * E], qkv[:, 2 * E:], bs, NHEAD, t, t, hd, nsplit=ns, f32=ns == 0, **sa)
        x = ops.add_layernorm(self.sa.out(_view3(att, bs, t, E), residual=xf), None, *self.norms[0], nsplit=ns)
        k = 1
        if self.ca is not None:
            if tc:
                kv = mem_kv.p if isinstance(mem_kv, ops.Act) else mem_kv
                att = ops.attention_tc(self.ca.q(x, want="p").p, 0, kv, 0, kv, E, bs, NHEAD, t, kv.rows, hd, nsplit=ns, **ca)
            else:
                tk = mem_kv.shape[1]
                assert mem_kv.is_contiguous()
                kv = mem_kv.view(bs * tk, 2 * E)
                q = self.ca.q(x).view(bs * t, E)
                att = ops.attention(q, kv[:, :E], kv[:, E:], bs, NHEAD, t, tk, hd, nsplit=ns, f32=ns == 0, **ca)
            x = ops.add_layernorm(self.ca.out(_view3(att, bs, t, E), residual=_f32(x)), None, *self.norms[1], nsplit=ns)
            k = 2
        h = self.l1(x, act=ops.ACT_RELU, want="p")
        want_ns = ns if "p" in want else 0
        y = ops.add_layernorm(self.l2(h, residual=_f32(x)), None, *self.norms[k], nsplit=want_ns, f32="f" in want or want_ns == 0)
        return y


def _attn_tc():
    """The tcgen05 attention kernel consumes two-plane fp16 operands: the fp16x3 engine."""
    return _STATE["nsplit"] == 2 and ops.plane_format() == "fp16"


def _window_of(x, j, bs):
    """Window j (clips j*bs .. (j+1)*bs) of a window-major hoisted tensor: fp32 tensor or plane Act."""
    if isinstance(x, ops.Act):
        pl = x.p
        return ops.Act(None, ops.Planes(pl.t[:, j * bs:(j + 1) * bs], pl.rows, pl.ch, 0))
    return x[j * bs:(j + 1) * bs]


def _view3(att, bs, t, E):
    """attention output (bs*t, E) fp32 tensor or Act -> (bs, t, E) view for the out-projection."""
    if isinstance(att, ops.Act):
        return ops.Act(None if att.f is None else att.f.view(bs, t, E), att.p)
    return att.view(bs, t, E)


class EmageEngine:
    """Packed EmageAudioModel (M.py:208-263)."""

    def __init__(self, sd, cfg):
        self.cfg = cfg
        E = self.E = int(cfg["hidden_size"])
        self.device = sd["mask_embedding"].device        # CUDA: enforced by the owning module and by ops._chk
        self.wav_face = _WavEncoder(sd, "audio_encoder_face")
        self.wav_body = _WavEncoder(sd, "audio_encoder_body")
        self.motion_encoder = _ConvStack(sd, "motion_encoder", "encoder", 3)            # M.py:227-231
        self.hint_face, self.hint_body = _MLP(sd, "bodyhints_face"), _MLP(sd, "bodyhints_body")
        af = int(cfg["audio_f"])
        wf, bf = sd["audio_face_motion_proj.weight"], sd["audio_face_motion_proj.bias"]
        self.face_mem_audio = _Linear(None, w=wf[:, :af], b=bf)       # audio half of the 512->768 proj (hoisted)
        self.face_mem_hint = _Linear(None, w=wf[:, af:], b=None)      # motion-hint half (in loop, accumulates)
        self.body_mem = _Linear(sd, "audio_body_motion_proj")
        self.moton_proj = _Linear(sd, "moton_proj")
        self.spk_face = sd["speaker_embedding_face.weight"].contiguous()
        self.spk_body = sd["speaker_embedding_body.weight"].contiguous()
        self.pe = sd["position_embeddings.pe"][0].contiguous()                         # (128, E)
        self.mask_embedding = sd["mask_embedding"].reshape(-1).contiguous()
        self.self_enc = _Layer(sd, "motion_self_encoder.layers.0", E, cross=False)
        self.cross = [_Layer(sd, f"audio_motion_cross_attn.layers.{i}", E, True) for i in range(8)]
        self.face_dec = [_Layer(sd, f"face_motion_decoder.layers.{i}", E, True) for i in range(4)]
        self.refine = {p: _Layer(sd, f"body_motion_decoder_{p}.layers.0", E, True) for p in PARTS[1:]}
        self.to_latent = {p: _MLP(sd, "motion2latent_" + p) for p in PARTS[1:]}
        self.out_proj = {p: _Linear(sd, "motion_out_proj_" + p) for p in PARTS[1:]}
        self.out_proj["face"] = _Linear(sd, "face_out_proj")
        self.cls = {p: _MLP(sd, "motion_cls_" + p) for p in PARTS[1:]}
        self.cls["face"] = _MLP(sd, "face_cls")
        self._fork_audio = _Fork(1)
        self._lane_forks = {}          # clip-group lane -> (face || body fork, refine-parts fork): side streams are per lane

    # ------------------------------------------------------------------------------------------------
    def audio_phase(self, audio, offset, a_ws, windows, n_samples, t, limits=None):
        """Everything that depends on audio only, for `windows` equally long slices per clip.
        Returns window-major tensors: face memory audio part (w*bs, t, E), body cross-attn K|V of the
        8 layers (list of (w*bs, tk, 2E)).  limits: a ragged batch's WavEncoder limits (RaggedLimits.wav)."""
        if wav_out_len(n_samples) < t:
            raise ValueError(f"audio slice yields {wav_out_len(n_samples)} frames < {t} motion frames")
        wl = {} if limits is None else {"limits": limits}

        def face():
            a_face = self.wav_face(audio, offset, a_ws, windows, n_samples, **wl)
            return self.face_mem_audio(a_face[:, :t])      # M.py:278-281 (the body stream is never truncated)

        def body():
            mem_body = self.body_mem(self.wav_body(audio, offset, a_ws, windows, n_samples, **wl), want="p" if _ns() else "f")
            return [layer.project_memory(mem_body) for layer in self.cross]

        kv, mem_face = self._fork_audio.run([body, face])
        return mem_face, kv

    def _forks(self, lane):
        if lane not in self._lane_forks:
            self._lane_forks[lane] = (_Fork(1), _Fork(2))
        return self._lane_forks[lane]

    def window(self, win_in, speaker_id_rows, mem_face_audio, kv_body, dest=None, use_audio=True, lane=0, limits=None):
        """One window of EmageAudioModel.forward (M.py:265-341) given the hoisted audio tensors.
        win_in (bs,t,337) is already mask-embedded.  speaker_id_rows = (spk_face_rows, spk_body_rows).
        dest: optional dict name -> (bs, t, 256) fp32 view the final GEMM of that output writes into (the window's rows
        of inference()'s accumulated outputs), so nothing is copied afterwards.
        limits: ragged batch - per-clip (rows, body memory keys, rows written to dest) of this window, int32 device
        tensors (RaggedLimits.window); None: every clip has t rows."""
        dest = dest or {}
        rows, tk, dest_rows = limits if limits is not None else (None, None, None)
        rl = {} if rows is None else {"row_limit": rows}
        self_kq = {} if rows is None else {"q_len": rows, "k_len": rows}
        cross_k = {} if rows is None else {"q_len": rows, "k_len": tk}
        out_rl = {} if rows is None else {"row_limit": dest_rows}
        fork_branch, fork_parts = self._forks(lane)
        # use_audio=False (training-time ablation, M.py:310-311): the body's audio cross-attention output is multiplied
        # by zero, i.e. motion_fea + 0 - the 8 cross layers are simply not run; the face branch still sees the audio.
        bs, t = (win_in.p.batch, win_in.p.rows) if isinstance(win_in, ops.Act) and win_in.f is None else _f32(win_in).shape[:2]
        E = self.E
        spk_f, spk_b = speaker_id_rows
        ns = _ns()
        hint = self.motion_encoder(win_in, want="p" if ns else "f", **rl)              # M.py:271

        def face_branch():                                                              # M.py:288-294
            hint_face = self.hint_face(hint, want="p" if ns else "f")
            mem_f = self.face_mem_hint(hint_face, residual=mem_face_audio, want="p" if ns else "f")
            x = ops.add_rows(None, self.pe, spk_f, ops.ROW_SPK, ops.ROW_PE, bs, t, E, nsplit=ns)
            for i, layer in enumerate(self.face_dec):
                x = layer(x, layer.project_memory(mem_f), want="fp" if i + 1 < len(self.face_dec) else "p", **self_kq)
            rec = self.out_proj["face"](x, want="fp", out=dest.get("rec_face"), **out_rl)
            return {"rec_face": _f32(rec), "cls_face": self.cls["face"](rec, out=dest.get("cls_face"), **out_rl)}

        def body_branch():                                                              # M.py:297-330
            hint_body = self.hint_body(hint, want="p" if ns else "f")
            x = ops.add_rows(self.moton_proj(hint_body), self.pe, spk_b, ops.ROW_PE, ops.ROW_SPK, bs, t, E, nsplit=ns)
            fea = self.self_enc(x, **self_kq)
            fea = ops.add_rows(fea, self.pe, spk_b, ops.ROW_SPK, ops.ROW_PE, bs, t, E, nsplit=ns)
            x = fea
            if use_audio:
                for i, (layer, kv) in enumerate(zip(self.cross, kv_body)):
                    x = layer(x, kv, want="fp" if i + 1 < len(self.cross) else "f", **cross_k)
                fea = ops.add2(_f32(fea), _f32(x), nsplit=ns, f32=ns == 0)
            else:
                fea = ops.add2(_f32(fea), torch.zeros_like(_f32(fea)), nsplit=ns, f32=ns == 0)
            lat = {p: self.to_latent[p](fea) for p in PARTS[1:]}
            others = {"upper": ("hands", "lower"), "hands": ("upper", "lower"), "lower": ("upper", "hands")}

            def refine(p):
                a, b = others[p]
                layer = self.refine[p]
                tgt = ops.add_rows(lat[p], self.pe, spk_b, ops.ROW_SPK, ops.ROW_NONE, bs, t, E, nsplit=ns)
                mem = ops.add2(lat[a], lat[b], nsplit=ns, f32=ns == 0)
                r = layer(tgt, layer.project_memory(mem), **self_kq)
                rec = self.out_proj[p](ops.add2(lat[p], r, nsplit=ns, f32=ns == 0), want="fp", out=dest.get("rec_" + p),
                                       **out_rl)
                return {"rec_" + p: _f32(rec), "cls_" + p: self.cls[p](rec, out=dest.get("cls_" + p), **out_rl)}

            out = {}
            for d in fork_parts.run([lambda p=p: refine(p) for p in PARTS[1:]]):
                out.update(d)
            return out

        body, face = fork_branch.run([body_branch, face_branch])
        body.update(face)
        return body

    def speaker_rows(self, speaker_id):
        """nn.Embedding lookup of the (bs,1) speaker ids (M.py:285-286): pure row gather."""
        ids = speaker_id.reshape(-1).to(torch.int64).contiguous()
        return ops.gather_rows(self.spk_face, ids), ops.gather_rows(self.spk_body, ids)


class VQEngine:
    """Packed EmageVQModel: four EmageVQVAEConv decoders/codebooks + the global EmageVAEConv
    (M.py:19-205)."""

    DIMS = {"face": 106, "upper": 78, "hands": 180, "lower": 61}

    def __init__(self, sds, cfgs):
        self.codebook, self.e2, self.decoder, self.encoder, self.vae_layers = {}, {}, {}, {}, {}
        for p in PARTS:
            sd, cfg = sds[p], cfgs[p]
            self.codebook[p] = sd["quantizer.embedding.weight"].contiguous()
            self.e2[p] = ops.row_sqnorm(self.codebook[p])
            self.decoder[p] = _ConvStack(sd, "decoder", "decoder", int(cfg["vae_layer"]))
            self.vae_layers[p] = int(cfg["vae_layer"])
            self._enc_args = None
        self.has_global = "global" in sds and sds["global"] is not None
        if self.has_global:
            n = int(cfgs["global"]["vae_layer"])
            self.global_enc = _ConvStack(sds["global"], "encoder", "encoder", n)
            self.global_dec = _ConvStack(sds["global"], "decoder", "decoder", n)
        self.device = self.codebook["face"].device
        self._forks = {}               # clip-group lane -> fork of the four part decoders

    def part_decode(self, p, index=None, latent=None, row_limit=None):
        """EmageVQVAEConv.decode / decode_from_latent (M.py:56-70) -> (pose features, indices).
        row_limit: per-clip frame counts of a ragged batch (int32 device tensor), None = all rows."""
        if index is None:                           # latent: (bs, t, 256), dense rows, any clip stride (a window's tail)
            index = ops.l2_argmin(latent, self.codebook[p], self.e2[p])
        if row_limit is None:
            return self.decoder[p](ops.gather_rows(self.codebook[p], index.contiguous(), nsplit=_ns())), index
        x = ops.gather_rows(self.codebook[p], index.contiguous(), nsplit=_ns(), row_limit=row_limit)
        return self.decoder[p](x, row_limit=row_limit), index

    def decode(self, index, latent, get_global_motion=False, ref_trans=None, lane=0, row_limit=None):
        """index/latent: dicts part -> tensor or None.  Returns the reference's 4-key dict (M.py:193).
        row_limit: per-clip frame counts of a ragged batch: every conv zeroes the frames beyond."""
        shape = next(t.shape[:2] for t in list(index.values()) + list(latent.values()) if t is not None)
        bs, t = int(shape[0]), int(shape[1])
        todo = [p for p in PARTS if index.get(p) is not None or latent.get(p) is not None]
        if lane not in self._forks:
            self._forks[lane] = _Fork(3)
        done = self._forks[lane].run([lambda p=p: self.part_decode(p, index.get(p), latent.get(p), row_limit=row_limit)[0]
                                      for p in todo])
        feats = dict(zip(todo, done))
        expression, aa, m4 = ops.pose_compose(feats.get("face"), feats.get("upper"), feats.get("hands"),
                                              feats.get("lower"), bs, t, self.device)
        trans = None
        if get_global_motion:
            lower_mix = feats.get("lower")
            if lower_mix is None:                   # M.py:174-178: identity rotations + zero trans/contact
                lower_mix = torch.zeros(bs, t, 61, device=self.device)
                lower_mix[:, :, 0:54:6] = 1.0
                lower_mix[:, :, 4:54:6] = 1.0
            trans = self.global_motion(lower_mix, ref_trans, row_limit=row_limit)
        return dict(expression=expression, all_motion4inference=m4, motion_axis_angle=aa, trans=trans)

    def global_motion(self, lower_mix, ref_trans, row_limit=None):
        """M.py:195-205."""
        rl = {} if row_limit is None else {"row_limit": row_limit}
        rec = self.global_dec(self.global_enc(lower_mix, **rl), **rl)
        bs = rec.shape[0]
        ref_trans = ref_trans.to(device=rec.device, dtype=torch.float32)
        if ref_trans.dim() == 2:                    # (n,3) -> every clip starts at row 0 (M.py:198-201)
            ref = ref_trans[0:1].expand(bs, 3)      # stride-0 view: the kernel takes the clip stride
        else:
            ref = ref_trans[:, 0]
            if ref.stride(1) != 1:
                ref = ref.contiguous()
        return ops.global_trans(rec, ref, 1 / 30)


def seed_decode_frames(cfg, vq):
    """Frames of a window's tail the in-loop VQ decode has to produce so that its last `seed_frames` outputs equal a
    decode of the whole window (M.py:411-418): the part decoders are stacks of k=3 convs - 2 ResBlocks (4 convs),
    vae_layer convs, 1 output conv - so an output frame sees +-(5 + vae_layer) latent frames (ADVICE r1: derived from
    the config instead of a constant 16)."""
    halo = 5 + max(vq.vae_layers.values())
    return int(cfg["seed_frames"]) + halo


def select_inputs(cfg, out, idx):
    """M.py:403-410 / T.py:34-42: latent for a part iff l?>0 and c?==0, class index iff c?>0."""
    index, latent = {}, {}
    for p, lk, ck in (("face", "lf", "cf"), ("upper", "lu", "cu"), ("hands", "lh", "ch"), ("lower", "ll", "cl")):
        latent[p] = out["rec_" + p] if cfg[lk] > 0 and cfg[ck] == 0 else None
        index[p] = idx[p] if cfg[ck] > 0 else None
    return index, latent


def window_plan(total_len, window, pre):
    """M.py:365-368,380-382,428-430 -> [(start, end, frames kept)]."""
    step = window - pre
    rounds, remain = (total_len - pre) // step, (total_len - pre) % step
    plan = [(i * step, i * step + window, step) for i in range(rounds)]
    if remain > pre:
        plan.append((rounds * step, rounds * step + pre + remain, pre + remain))
    return plan


def run_inference(engine: EmageEngine, vq: VQEngine, audio, speaker_id, masked_motion=None, mask=None):
    """EmageAudioModel.inference (M.py:343-490)."""
    cfg = engine.cfg
    dev = engine.device
    audio = audio.to(device=dev, dtype=torch.float32).contiguous()
    bs, n = audio.shape
    length = n * 30 // 16000                                                             # M.py:345
    window, pre = int(cfg["pose_length"]), int(cfg["seed_frames"])
    ch = int(cfg["pose_dims"]) + 7
    # No masked_motion / mask given (the demo's call): the defaults - identity rotations (rot6d [1,0,0,0,1,0]) + zero
    # trans / contact, everything masked (M.py:369-377) - are generated inside window_input, no tensors are built.
    motion = full_mask = None
    if masked_motion is not None or mask is not None:
        motion = torch.zeros(bs, length, ch, device=dev)
        motion[:, :, 0:ch - 7:6] = 1.0
        motion[:, :, 4:ch - 7:6] = 1.0
        if masked_motion is not None:
            motion[:, :masked_motion.shape[1]] = masked_motion.to(dev)
        full_mask = torch.ones(bs, length, ch, device=dev)
        if mask is not None:
            full_mask[:, :mask.shape[1]] = mask.to(dev)
    plan = window_plan(length, window, pre)
    spf = 16000 // 30                                                                    # 533, M.py:393
    if not plan:
        raise RuntimeError("audio too short: no window to generate (reference torch.cat of an empty list fails too)")
    spk = engine.speaker_rows(speaker_id.to(dev))

    # ---- hoisted audio phase: full windows as one batch, tail window separately ----
    n_full = sum(1 for s, e, _ in plan if e - s == window)
    groups = []
    if n_full:
        groups.append((0, n_full, window))
    if len(plan) > n_full:
        groups.append((n_full, 1, plan[-1][1] - plan[-1][0]))
    hoisted = {}
    for first, count, t in groups:
        s0 = plan[first][0]
        mem_face, kv = engine.audio_phase(audio, s0 * spf, (window - pre) * spf, count, t * spf, t)
        E = engine.E
        mem_face = mem_face.view(count, bs, t, E)                 # window-major: each window is contiguous
        for j in range(count):
            hoisted[first + j] = (mem_face[j], [_window_of(k, j, bs) for k in kv])

    out_len = sum(k for _, _, k in plan)
    # Every window writes its t frames straight into the accumulated outputs at its offset; the `pre` frames beyond the
    # `keep` it contributes (M.py:419-426) are overwritten by the next window.  Only a full-length LAST window would
    # spill past the end: `pad` spare rows take that, and the result is the dense [:out_len] prefix (a copy only then).
    pad = max(0, max(off_t for off_t in [sum(k for _, _, k in plan[:i]) + (e - s) for i, (s, e, _) in enumerate(plan)]) - out_len)
    acc = {k + p: torch.empty(bs, out_len + pad, 256, device=dev) for k in ("rec_", "cls_") for p in PARTS}
    # Clips are independent, and one window is a chain of ~150 dependent kernels whose GEMMs fill 48-288 of the 148 SMs:
    # the clip batch is therefore split into `groups` lanes that run their window loops on separate streams, so that
    # one lane's launch gaps, drains and epilogue tails are filled by the other lane's thread blocks (the hoisted audio
    # phase above and the final decode stay batched).  Per-clip results do not depend on the grouping.
    n_groups = max(1, min(int(_STATE.get("groups", 1)), bs // 8)) if torch.cuda.is_available() else 1
    bounds = [bs * g // n_groups for g in range(n_groups + 1)]

    def sl(x, g0, g1):                # clips g0..g1 of a (clips, ...) tensor, plane Act or None
        if x is None:
            return None
        if isinstance(x, ops.Act):
            pl = x.p
            return ops.Act(None if x.f is None else x.f[g0:g1], None if pl is None else ops.Planes(pl.t[:, g0:g1], pl.rows, pl.ch, 0))
        return x[g0:g1]

    def run_lane(lane):
        g0, g1 = bounds[lane], bounds[lane + 1]
        nb = g1 - g0
        spk_l = (spk[0][g0:g1], spk[1][g0:g1])
        seed = None                   # first window: the seed is motion[:, :pre] itself (M.py:379) - window_input keeps it
        off = 0
        for wi, (s, e, keep) in enumerate(plan):
            t = e - s
            win_in = ops.window_input(sl(motion, g0, g1), sl(full_mask, g0, g1), seed, engine.mask_embedding, s, t, pre,
                                      nsplit=_ns(), f32=_ns() == 0, shape=(nb, length, ch))
            mem_face, kv = hoisted[wi]
            out = engine.window(win_in, spk_l, sl(mem_face, g0, g1), [sl(k, g0, g1) for k in kv],
                                dest={k: v[g0:g1, off:off + t] for k, v in acc.items()}, lane=lane)
            off += keep
            if wi + 1 < len(plan):                                                       # seed for the next window
                nd = min(t, seed_decode_frames(cfg, vq))
                tail = {k: v[:, t - nd:] for k, v in out.items()}                        # strided views, read in place
                idx = {p: ops.row_argmax(tail["cls_" + p]) for p in PARTS}               # M.py:398-401
                index, latent = select_inputs(cfg, tail, idx)
                dec = vq.decode(index, latent, lane=lane)
                seed = dec["all_motion4inference"][:, nd - pre:]                         # M.py:418
        return None

    if n_groups == 1:
        run_lane(0)
    else:
        if getattr(engine, "_fork_lanes", None) is None or engine._fork_lanes.n_side != n_groups - 1:
            engine._fork_lanes = _Fork(n_groups - 1)
        engine._fork_lanes.run([lambda lane=lane: run_lane(lane) for lane in range(n_groups)])
    if pad:
        acc = {k: v[:, :out_len].contiguous() for k, v in acc.items()}
    return acc


# ------------------------------------------------------------------------------------------------------
# Ragged batches: clips of different lengths in one batched schedule
# ------------------------------------------------------------------------------------------------------


class RaggedPlan:
    """Per-clip geometry of a ragged batch (host only).  Every clip is laid out at one capacity - `windows` windows of
    `window` rows for each of `batch` clips - and the int32 tables below say which rows of each (window, clip) are real.
    Window j of every clip starts at frame j*step and audio sample j*step*spf, as in run_inference().

      win_rows (W, B)      rows of clip b's window j: `window` for a full window, pre + remain for its tail window,
                           0 where the clip has no window j (window_plan, M.py:365-368)
      n_valid  (W, B)      audio samples of that window's slice: win_rows * spf
      wav_rows (6, W, B)   valid rows after each WavEncoder block (wav_block_lens of n_valid; 0 for empty slices)
      body_keys (W, B)     body cross-attention keys = wav_out_len(n_valid): the body stream is never truncated
                           (M.py:278-281), so a tail of T <= 25 rows has T + 1 keys
      dest_rows (W, B)     rows the window writes into the accumulated outputs: win_rows, -1 (nothing) where empty
      out_len  (B,)        emitted frames per clip
    """

    def __init__(self, n_samples, window, pre, batch=None, windows=None):
        n_samples = [int(n) for n in n_samples]
        self.window, self.pre, self.step, self.spf = window, pre, window - pre, 16000 // 30
        plans = [window_plan(n * 30 // 16000, window, pre) for n in n_samples]                  # M.py:345
        if any(not p or p[0][0] < 0 for p in plans):              # (fewer frames than `pre`: a window before frame 0)
            raise RuntimeError("audio too short: no window to generate (reference torch.cat of an empty list fails too)")
        self.batch = len(n_samples) if batch is None else int(batch)
        self.windows = max(len(p) for p in plans) if windows is None else int(windows)
        if len(n_samples) > self.batch or max(len(p) for p in plans) > self.windows:
            raise ValueError(f"{len(n_samples)} clips / {max(len(p) for p in plans)} windows exceed the capacity "
                             f"of {self.batch} clips x {self.windows} windows")
        W, B = self.windows, self.batch
        self.win_rows = np.zeros((W, B), np.int32)
        self.out_len = np.zeros(B, np.int32)
        for b, plan in enumerate(plans):
            for j, (s, e, _) in enumerate(plan):
                assert s == j * self.step
                self.win_rows[j, b] = e - s
            self.out_len[b] = sum(k for _, _, k in plan)
        self.n_valid = self.win_rows * self.spf
        self.wav_rows = np.zeros((len(WAV_BLOCKS), W, B), np.int32)
        for j in range(W):
            for b in range(B):
                if self.win_rows[j, b]:
                    self.wav_rows[:, j, b] = wav_block_lens(int(self.n_valid[j, b]))
        self.body_keys = self.wav_rows[-1].copy()
        self.dest_rows = np.where(self.win_rows > 0, self.win_rows, -1).astype(np.int32)
        self.n_clips = len(n_samples)

    @property
    def capacity_frames(self):
        return self.windows * self.step + self.pre

    @property
    def capacity_samples(self):
        """Audio samples the windows read: a clip's samples beyond this (the fraction of a frame after its last frame,
        or the frames of a dropped tail, M.py:380-382) are never part of any window."""
        return ((self.windows - 1) * self.step + self.window) * self.spf

    def tables(self):
        """name -> int32 array, in the layout RaggedLimits keeps on the device (slices window-major)."""
        W, B = self.windows, self.batch
        return {"n_valid": self.n_valid.reshape(W * B), "wav_rows": self.wav_rows.reshape(-1, W * B),
                "win_rows": self.win_rows, "body_keys": self.body_keys, "dest_rows": self.dest_rows,
                "out_len": self.out_len}


class RaggedLimits:
    """The tables of a RaggedPlan as int32 device tensors, the per-clip limit arguments of the `_rl` kernels.  All tables
    are views of one device buffer, so a plan loads with one host -> device copy; they keep their addresses across
    load() calls, so a graph captured with them reads whatever was loaded last."""

    def __init__(self, plan: RaggedPlan, device):
        tables = plan.tables()
        self.buf = torch.empty(sum(v.size for v in tables.values()), dtype=torch.int32, device=device)
        self.t, off = {}, 0
        for k, v in tables.items():
            self.t[k] = self.buf[off:off + v.size].view(v.shape)
            off += v.size
        self.windows, self.batch = plan.windows, plan.batch
        self.load(plan)

    def load(self, plan: RaggedPlan):
        assert (plan.windows, plan.batch) == (self.windows, self.batch)
        host = np.concatenate([v.ravel() for v in plan.tables().values()]).astype(np.int32)
        self.buf.copy_(torch.from_numpy(host))

    @property
    def wav(self):
        return self.t["n_valid"], list(self.t["wav_rows"])

    def window(self, j, g0, g1):
        return self.t["win_rows"][j, g0:g1], self.t["body_keys"][j, g0:g1], self.t["dest_rows"][j, g0:g1]

    @property
    def out_len(self):
        return self.t["out_len"]


def run_inference_ragged(engine: EmageEngine, vq: VQEngine, audio_padded, limits: RaggedLimits, speaker_id):
    """run_inference() for a ragged batch laid out at capacity: audio_padded (B, >= capacity samples), zero beyond
    each clip; limits = the batch's RaggedLimits.  Returns the accumulated rec_* / cls_* outputs (B, capacity frames,
    256): clip b's outputs are its first out_len[b] rows, equal to run_inference() of that clip alone."""
    cfg = engine.cfg
    dev = engine.device
    window, pre = int(cfg["pose_length"]), int(cfg["seed_frames"])
    step, spf = window - pre, 16000 // 30
    ch = int(cfg["pose_dims"]) + 7
    W, B = limits.windows, limits.batch
    audio = audio_padded.to(device=dev, dtype=torch.float32).contiguous()
    assert audio.shape[0] == B and audio.shape[1] >= ((W - 1) * step + window) * spf, audio.shape
    spk = engine.speaker_rows(speaker_id.to(dev))
    frames = W * step + pre

    # ---- hoisted audio phase: all W x B slices as one window-major batch at `window` rows ----
    mem_face, kv = engine.audio_phase(audio, 0, step * spf, W, window * spf, window, limits=limits.wav)
    mem_face = mem_face.view(W, B, window, engine.E)
    # Zeroed (memset, no kernel): rows no window writes stay finite for the full-length argmax and decode.
    acc = {}
    for k in ("rec_", "cls_"):
        for p in PARTS:
            acc[k + p] = torch.empty(B, frames, 256, device=dev)
            if acc[k + p].is_cuda:
                _lib.call("pm_memset_async", acc[k + p].data_ptr(), 0, acc[k + p].numel() * 4, ops._stream())
            else:
                acc[k + p].zero_()
    n_groups = max(1, min(int(_STATE.get("groups", 1)), B // 8)) if torch.cuda.is_available() else 1
    bounds = [B * g // n_groups for g in range(n_groups + 1)]

    def sl(x, g0, g1):
        if isinstance(x, ops.Act):
            pl = x.p
            return ops.Act(None if x.f is None else x.f[g0:g1], None if pl is None else ops.Planes(pl.t[:, g0:g1], pl.rows, pl.ch, 0))
        return x[g0:g1]

    def run_lane(lane):
        g0, g1 = bounds[lane], bounds[lane + 1]
        nb = g1 - g0
        spk_l = (spk[0][g0:g1], spk[1][g0:g1])
        seed = None
        for j in range(W):
            lim = limits.window(j, g0, g1)
            win_in = ops.window_input(None, None, seed, engine.mask_embedding, j * step, window, pre, nsplit=_ns(),
                                      f32=_ns() == 0, shape=(nb, frames, ch), row_limit=lim[0])
            out = engine.window(win_in, spk_l, mem_face[j][g0:g1], [sl(_window_of(k, j, B), g0, g1) for k in kv],
                                dest={k: v[g0:g1, j * step:j * step + window] for k, v in acc.items()}, lane=lane,
                                limits=lim)
            if j + 1 < W:                     # seed for the next window; only clips whose window j is full continue
                nd = min(window, seed_decode_frames(cfg, vq))
                tail = {k: v[:, window - nd:] for k, v in out.items()}
                idx = {p: ops.row_argmax(tail["cls_" + p]) for p in PARTS}
                index, latent = select_inputs(cfg, tail, idx)
                dec = vq.decode(index, latent, lane=lane)
                seed = dec["all_motion4inference"][:, nd - pre:]

    if n_groups == 1:
        run_lane(0)
    else:
        if getattr(engine, "_fork_lanes", None) is None or engine._fork_lanes.n_side != n_groups - 1:
            engine._fork_lanes = _Fork(n_groups - 1)
        engine._fork_lanes.run([lambda lane=lane: run_lane(lane) for lane in range(n_groups)])
    return acc
