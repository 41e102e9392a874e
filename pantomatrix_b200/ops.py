"""Thin torch-tensor wrappers over the C ABI (include/pm_emage.h).

torch is used only for device memory (torch.empty), the current CUDA stream and tensor views; every
arithmetic op of the hot path is a kernel of libpm_emage.so.  All functions require CUDA tensors and
raise (PmError) on any failure - there is no fallback.
"""
from __future__ import annotations

import math

import torch

from . import _lib

ACT_NONE, ACT_RELU, ACT_LEAKY = 0, 1, 2
ROW_NONE, ROW_PE, ROW_SPK = 0, 1, 2

# number of kernel launches issued through this module (bench.py reports it as gpu_launches)
launch_count = 0

# Element format of the tensor-core operand planes: bf16 (default) or IEEE fp16.  Two fp16 planes (3 products)
# match three bf16 planes (6 products) in accuracy while magnitudes stay below 65504 (include/pm_emage.h).
FMT_F16 = 0x100
# fp16 activation planes hold F16_ACT_SCALE * x (csrc/pm_common.cuh PM_F16_ACT_SCALE: the tensor core flushes fp16
# subnormal operands, the exact pre-scale keeps second planes normal down to |x| = 2^-9); PackedW.acc_scale undoes it.
F16_ACT_SCALE = 64.0
_PLANE_DTYPE = torch.bfloat16


def set_plane_format(name: str) -> None:
    global _PLANE_DTYPE
    _PLANE_DTYPE = {"bf16": torch.bfloat16, "fp16": torch.float16}[name]


def plane_format() -> str:
    return "fp16" if _PLANE_DTYPE == torch.float16 else "bf16"


def _fmt_bit(t) -> int:
    return FMT_F16 if t.dtype == torch.float16 else 0


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t) -> int | None:
    return None if t is None else t.data_ptr()


def _chk(t: torch.Tensor, dtype=torch.float32):
    if not t.is_cuda:
        raise _lib.PmError("pantomatrix_b200 ops need CUDA tensors (no CPU fallback)")
    if t.dtype != dtype:
        raise _lib.PmError(f"expected {dtype}, got {t.dtype}")
    if t.dim() and t.stride(-1) != 1 and t.shape[-1] != 1:
        raise _lib.PmError("innermost dimension must be contiguous")
    return t


def _call(name, *args):
    global launch_count
    launch_count += 1
    _lib.call(name, *args)


def _bs_ld(t: torch.Tensor):
    """(batch stride, row stride) in elements of a (batch, rows, ch) view."""
    return (t.stride(0) if t.shape[0] > 1 else t.shape[1] * t.stride(1)), t.stride(1)


def tapgemm(a, w, bias, *, rows_out=None, stride=1, pad=0, act=ACT_NONE, slope=0.0, residual=None, out=None,
            row_limit=None):
    """out[b,l,:] = act(bias + sum_t A[b, l*stride+t-pad, :] @ W[t].T + residual[b,l,:]).

    a: (batch, rows_in, cin); w: (taps, cout, cin) contiguous; returns (batch, rows_out, cout).
    row_limit: optional int32 device tensor (batch,) - ragged batch: rows l >= row_limit[b] are written as 0
    (a negative limit: clip b is not written)."""
    _chk(a), _chk(w)
    batch, rows_in, cin = a.shape
    taps, cout, cin_w = w.shape
    assert cin_w == cin and w.is_contiguous(), (w.shape, a.shape)
    if rows_out is None:
        rows_out = (rows_in + 2 * pad - taps) // stride + 1
    if out is None:
        out = torch.empty(batch, rows_out, cout, device=a.device, dtype=torch.float32)
    else:
        assert out.shape == (batch, rows_out, cout), (out.shape, (batch, rows_out, cout))
    _chk(out)
    if residual is not None:
        _chk(residual)
        assert residual.shape == out.shape
    # a Linear (taps == 1, no padding) over contiguous batches is one tall matrix: better tile use
    if (taps == 1 and pad == 0 and stride == 1 and batch > 1 and a.stride(0) == rows_in * a.stride(1)
            and out.stride(0) == rows_out * out.stride(1)
            and (residual is None or residual.stride(0) == rows_out * residual.stride(1))):
        a = a.reshape(1, batch * rows_in, cin) if a.is_contiguous() else a.as_strided(
            (1, batch * rows_in, cin), (0, a.stride(1), 1), a.storage_offset())
        flat = lambda t: t.as_strided((1, batch * rows_out, cout), (0, t.stride(1), 1), t.storage_offset())
        out_v = flat(out)
        res_v = flat(residual) if residual is not None else None
        batch_k, rows_in_k, rows_out_k = 1, batch * rows_in, batch * rows_out
        rows_per_clip = rows_out
    else:
        out_v, res_v, batch_k, rows_in_k, rows_out_k = out, residual, batch, rows_in, rows_out
        rows_per_clip = 0
    a_bs, lda = _bs_ld(a)
    o_bs, ldo = _bs_ld(out_v)
    r_bs, ldr = _bs_ld(res_v) if res_v is not None else (0, 0)
    if row_limit is None:
        _call("pm_tapgemm_f32", a.data_ptr(), a_bs, lda, batch_k, rows_in_k, cin,
              w.data_ptr(), _ptr(bias), taps, stride, pad, rows_out_k, cout,
              _ptr(res_v), r_bs, ldr, act, float(slope), out_v.data_ptr(), o_bs, ldo, _stream())
    else:
        _chk_limit(row_limit, batch)
        _call("pm_tapgemm_f32_rl", a.data_ptr(), a_bs, lda, batch_k, rows_in_k, cin,
              w.data_ptr(), _ptr(bias), taps, stride, pad, rows_out_k, cout,
              _ptr(res_v), r_bs, ldr, act, float(slope), out_v.data_ptr(), o_bs, ldo, row_limit.data_ptr(), rows_per_clip,
              _stream())
    return out


def _chk_limit(t, n):
    """A per-clip limit table: int32 device tensor of at least n entries, read by the kernel."""
    _chk(t, torch.int32)
    assert t.dim() == 1 and t.is_contiguous() and t.numel() >= n, (t.shape, n)


def wav_stem(audio, a_bs, a_ws, batch, windows, n_samples, w1, b1, wd, bd, *, stride, pad, slope, offset=0, nsplit=0,
             n_valid=None):
    """First WavEncoder block's two convolutions on the raw waveform.  `audio` is the flat (bs, n)
    tensor; sequence (b, w) starts at element offset + b*a_bs + w*a_ws and is n_samples long.
    Returns (y1, sc): y1 as fp32 tensor (nsplit 0) or as the operand Planes of the conv that follows.
    n_valid: optional int32 device tensor (windows*batch,), window-major - ragged batch: sequence w*batch + b holds only
    n_valid samples (later ones read as 0) and the rows it does not yield are written as 0."""
    _chk(audio)
    cout, ks = w1.shape
    rows_out = (n_samples + 2 * pad - ks) // stride + 1
    sc = torch.empty(batch * windows, rows_out, cout, device=audio.device, dtype=torch.float32)
    if nsplit:
        y1 = _new_planes(nsplit, (batch * windows, rows_out), cout, audio.device)
        y_ptr, pa = 0, (y1.t.data_ptr(), y1.t.stride(0), y1.t.stride(2), nsplit | _fmt_bit(y1.t))
    else:
        y1 = torch.empty_like(sc)
        y_ptr, pa = y1.data_ptr(), (0, 0, 0, 0)
    if n_valid is None:
        _call("pm_wav_stem_f32", audio.data_ptr() + 4 * offset, a_bs, a_ws, batch, windows, n_samples,
              w1.data_ptr(), b1.data_ptr(), wd.data_ptr(), bd.data_ptr(), cout, ks, stride, pad, rows_out,
              float(slope), y_ptr, sc.data_ptr(), *pa, _stream())
    else:
        _chk_limit(n_valid, batch * windows)
        _call("pm_wav_stem_rl", audio.data_ptr() + 4 * offset, a_bs, a_ws, batch, windows, n_samples,
              w1.data_ptr(), b1.data_ptr(), wd.data_ptr(), bd.data_ptr(), cout, ks, stride, pad, rows_out,
              float(slope), y_ptr, sc.data_ptr(), *pa, n_valid.data_ptr(), _stream())
    return y1, sc


class Act:
    """One activation as fp32 tensor (`f`) and/or split-bf16 planes (`p`); either may be None."""
    __slots__ = ("f", "p")

    def __init__(self, f=None, p=None):
        self.f, self.p = f, p


def _new_planes(nsplit, lead_shape, ch, device, slack_rows=0, dtype=None):
    """Planes for an activation of shape (*lead_shape, ch); lead_shape = (batch, rows)."""
    batch, rows = lead_shape
    dtype = dtype or _PLANE_DTYPE
    ld = _round_up(ch, 8)
    if slack_rows:
        buf = torch.empty(nsplit, batch * rows + slack_rows, ld, device=device, dtype=dtype)
        if buf.is_cuda:
            for i in range(nsplit):               # cudaMemsetAsync: a memset node under graph capture, not a kernel
                _lib.call("pm_memset_async", buf[i, batch * rows:].data_ptr(), 0, slack_rows * ld * buf.element_size(), _stream())
        else:
            buf[:, batch * rows:].zero_()
        t = buf[:, :batch * rows].view(nsplit, batch, rows, ld)
    else:
        t = torch.empty(nsplit, batch, rows, ld, device=device, dtype=dtype)
    return Planes(t, rows, ch, slack_rows)


def _pargs(pl):
    if pl is None:
        return None, 0, 0, 0
    return pl.t.data_ptr(), pl.t.stride(0), pl.t.stride(2), pl.t.shape[0] | _fmt_bit(pl.t)


def _result(f, pl, nsplit):
    return f if nsplit == 0 else Act(f, pl)


def add_layernorm(x, r, gamma, beta, eps=1e-5, nsplit=0, f32=True):
    _chk(x)
    assert x.is_contiguous() and (r is None or (r.is_contiguous() and r.shape == x.shape))
    ch = x.shape[-1]
    rows = x.numel() // ch
    out = torch.empty_like(x) if (f32 or not nsplit) else None
    pl = _new_planes(nsplit, (x.shape[0], rows // x.shape[0]), ch, x.device) if nsplit else None
    _call("pm_add_layernorm_f32", x.data_ptr(), _ptr(r), gamma.data_ptr(), beta.data_ptr(), _ptr(out),
          rows, ch, float(eps), *_pargs(pl), _stream())
    return _result(out, pl, nsplit)


def attention(q, k, v, batch, heads, tq, tk, head_dim, nsplit=0, f32=True, q_len=None, k_len=None):
    """q: (batch*tq, >=heads*head_dim) view, k/v: (batch*tk, ...) views (column slices allowed).
    q_len / k_len: optional int32 device tensors (batch,) - ragged batch: keys >= k_len[b] get probability 0, query rows
    >= q_len[b] (all rows when k_len[b] == 0) are written as 0.  Both or neither."""
    for t in (q, k, v):
        _chk(t)
    E = heads * head_dim
    out = torch.empty(batch * tq, E, device=q.device, dtype=torch.float32) if (f32 or not nsplit) else None
    pl = _new_planes(nsplit, (batch, tq), E, q.device) if nsplit else None
    if k_len is None:
        _call("pm_attention_f32", q.data_ptr(), q.stride(0), k.data_ptr(), k.stride(0), v.data_ptr(), v.stride(0),
              _ptr(out), E, batch, heads, tq, tk, head_dim, *_pargs(pl), _stream())
    else:
        _chk_limit(q_len, batch), _chk_limit(k_len, batch)
        _call("pm_attention_f32_rl", q.data_ptr(), q.stride(0), k.data_ptr(), k.stride(0), v.data_ptr(), v.stride(0),
              _ptr(out), E, batch, heads, tq, tk, head_dim, *_pargs(pl), q_len.data_ptr(), k_len.data_ptr(), _stream())
    return _result(out, pl, nsplit)


def attention_tc(q, q_col0, k, k_col0, v, v_col0, batch, heads, tq, tk, head_dim, nsplit=2, f32=False, q_len=None,
                 k_len=None):
    """Attention on the tcgen05 tensor cores (fp16x3 engine).  q / k / v: two-plane fp16 Planes whose columns
    [*_col0 + h*head_dim, ...) hold head h (the packed q|k|v or k|v projection output is passed as is).
    q_len / k_len: per-clip counts as in attention()."""
    for pl, rows in ((q, tq), (k, tk), (v, tk)):
        assert pl.t.dtype == torch.float16 and pl.t.shape[0] == 2 and pl.t.shape[1] == batch and pl.rows == rows, \
            "attention_tc needs two-plane fp16 operands of (batch, rows, ch)"
    E = heads * head_dim
    dev = q.t.device
    out = torch.empty(batch * tq, E, device=dev, dtype=torch.float32) if (f32 or not nsplit) else None
    pl = _new_planes(nsplit, (batch, tq), E, dev, dtype=torch.float16) if nsplit else None
    if k_len is None:
        _call("pm_attention_tc",
              q.t.data_ptr(), q.t.stride(0), q.t.stride(1), q.t.stride(2), q.ch, q_col0,
              k.t.data_ptr(), k.t.stride(0), k.t.stride(1), k.t.stride(2), k.ch, k_col0,
              v.t.data_ptr(), v.t.stride(0), v.t.stride(1), v.t.stride(2), v.ch, v_col0,
              _ptr(out), E, batch, heads, tq, tk, head_dim, *_pargs(pl), _stream())
    else:
        _chk_limit(q_len, batch), _chk_limit(k_len, batch)
        _call("pm_attention_tc_rl",
              q.t.data_ptr(), q.t.stride(0), q.t.stride(1), q.t.stride(2), q.ch, q_col0,
              k.t.data_ptr(), k.t.stride(0), k.t.stride(1), k.t.stride(2), k.ch, k_col0,
              v.t.data_ptr(), v.t.stride(0), v.t.stride(1), v.t.stride(2), v.ch, v_col0,
              _ptr(out), E, batch, heads, tq, tk, head_dim, *_pargs(pl), q_len.data_ptr(), k_len.data_ptr(), _stream())
    return _result(out, pl, nsplit)


def add_rows(x, pe, spk, first, second, batch, rows, ch, nsplit=0, f32=True):
    dev = (pe if pe is not None else spk).device
    out = torch.empty(batch, rows, ch, device=dev, dtype=torch.float32) if (f32 or not nsplit) else None
    if x is not None:
        _chk(x)
        assert x.is_contiguous() and x.numel() == batch * rows * ch
    pl = _new_planes(nsplit, (batch, rows), ch, dev) if nsplit else None
    _call("pm_add_rows_f32", _ptr(x), _ptr(pe), _ptr(spk), first, second, _ptr(out), batch, rows, ch, *_pargs(pl), _stream())
    return _result(out, pl, nsplit)


def add2(a, b, nsplit=0, f32=True):
    _chk(a), _chk(b)
    assert a.is_contiguous() and b.is_contiguous() and a.shape == b.shape
    out = torch.empty_like(a) if (f32 or not nsplit) else None
    ch = a.shape[-1]
    pl = _new_planes(nsplit, (a.shape[0], a.numel() // ch // a.shape[0]), ch, a.device) if nsplit else None
    _call("pm_add2_f32", a.data_ptr(), b.data_ptr(), _ptr(out), a.numel(), ch, *_pargs(pl), _stream())
    return _result(out, pl, nsplit)


def window_input(motion, mask, seed, mask_embedding, start, win_len, pre, nsplit=0, f32=True, shape=None, row_limit=None):
    """motion / mask: (batch, total_len, ch) or None = inference()'s defaults (then `shape` = (batch, total_len, ch));
    seed: (batch, pre, ch) view with dense rows (any clip stride), None when pre == 0.
    row_limit: optional int32 device tensor (batch,) - ragged batch: rows >= row_limit[b] are written as 0."""
    batch, total_len, ch = motion.shape if motion is not None else shape
    for t in (motion, mask):
        if t is not None:
            _chk(t)
            assert t.is_contiguous() and t.shape == (batch, total_len, ch)
    seed_bs = 0
    if seed is not None:
        _chk(seed)
        assert seed.shape == (batch, pre, ch) and (pre <= 1 or seed.stride(1) == ch)
        seed_bs = seed.stride(0)
    dev = mask_embedding.device
    out = torch.empty(batch, win_len, ch, device=dev, dtype=torch.float32) if (f32 or not nsplit) else None
    pl = _new_planes(nsplit, (batch, win_len), ch, dev) if nsplit else None
    if row_limit is None:
        _call("pm_window_input_f32", _ptr(motion), _ptr(mask), _ptr(seed), mask_embedding.data_ptr(),
              _ptr(out), batch, total_len, start, win_len, pre, ch, seed_bs, *_pargs(pl), _stream())
    else:
        _chk_limit(row_limit, batch)
        _call("pm_window_input_rl", _ptr(motion), _ptr(mask), _ptr(seed), mask_embedding.data_ptr(),
              _ptr(out), batch, total_len, start, win_len, pre, ch, seed_bs, *_pargs(pl), row_limit.data_ptr(), _stream())
    return _result(out, pl, nsplit)


def _batched_rows(x, ld):
    """(rows, rows_per_batch, batch stride) of a (rows, ch) matrix or a (batch, rows, ch) view whose rows are `ld` apart."""
    if x.dim() == 2:
        assert x.stride(0) == ld
        return x.shape[0], 0, 0
    assert x.dim() == 3 and (x.shape[1] == 1 or x.stride(1) == ld)
    return x.shape[0] * x.shape[1], x.shape[1], x.stride(0)


def l2_argmin(z, codebook, e2, engine="auto", max_ctas=0):
    """fp32 argmin_k |z - e_k|^2, first minimum wins.  engine: "auto" (the product path: tcgen05 screen + exact fp32
    re-scoring for 256-code codebooks, fp32 SIMT otherwise), "tc" or "simt" (tests / microbenchmarks)."""
    _chk(z), _chk(codebook), _chk(e2)
    assert codebook.is_contiguous()
    n_codes, e_dim = codebook.shape
    if z.dim() > 3:
        z = z.reshape(-1, e_dim)
    rows, rpb, z_bs = _batched_rows(z, e_dim)      # (rows, 256) or a (batch, rows, 256) view, e.g. the tail of a window
    idx = torch.empty(z.shape[:-1], device=z.device, dtype=torch.int64)
    if engine == "tc":
        _call("pm_l2_argmin_tc", z.data_ptr(), rows, rpb, z_bs, codebook.data_ptr(), e2.data_ptr(), n_codes, e_dim,
              idx.data_ptr(), int(max_ctas), _stream())
    elif engine == "simt":
        _call("pm_l2_argmin_simt_f32", z.data_ptr(), rows, rpb, z_bs, codebook.data_ptr(), e2.data_ptr(), n_codes, e_dim,
              idx.data_ptr(), _stream())
    else:
        _call("pm_l2_argmin_f32", z.data_ptr(), rows, rpb, z_bs, codebook.data_ptr(), e2.data_ptr(), n_codes, e_dim,
              idx.data_ptr(), _stream())
    return idx


def row_argmax(x, nonfinite=None):
    """First argmax over the last dim of a (rows, ch) matrix or a (batch, rows, ch) view (any clip stride).
    nonfinite: optional int32[1] device flag, set to 1 when a NaN / inf is read (never cleared here)."""
    _chk(x)
    ch = x.shape[-1]
    if x.dim() > 3:
        x = x.reshape(-1, ch)
    ld = x.stride(-2) if x.shape[-2] > 1 else ch
    rows, rpb, x_bs = _batched_rows(x, ld)
    idx = torch.empty(x.shape[:-1], device=x.device, dtype=torch.int64)
    _call("pm_row_argmax_f32", x.data_ptr(), rows, ch, ld, rpb, x_bs, idx.data_ptr(), _ptr(nonfinite), _stream())
    return idx


def zero_flag(device):
    """int32[1] device flag cleared by a memset node (no kernel)."""
    flag = torch.empty(1, device=device, dtype=torch.int32)
    _lib.call("pm_memset_async", flag.data_ptr(), 0, 4, _stream())
    return flag


def gather_rows(codebook, index, nsplit=0, f32=True, row_limit=None):
    """row_limit: optional int32 device tensor (index.shape[0],) for a (clips, rows) index - ragged batch: rows
    >= row_limit[clip] are written as 0."""
    _chk(codebook), _chk(index, torch.int64)
    assert index.is_contiguous()
    ch = codebook.shape[1]
    out = torch.empty(*index.shape, ch, device=codebook.device, dtype=torch.float32) if (f32 or not nsplit) else None
    pl = None
    if nsplit:
        lead = (index.shape[0], index.numel() // index.shape[0]) if index.dim() > 1 else (1, index.numel())
        pl = _new_planes(nsplit, lead, ch, codebook.device)
    if row_limit is None:
        _call("pm_gather_rows_f32", codebook.data_ptr(), codebook.shape[0], index.data_ptr(), index.numel(), ch, _ptr(out),
              *_pargs(pl), _stream())
    else:
        assert index.dim() == 2
        _chk_limit(row_limit, index.shape[0])
        _call("pm_gather_rows_rl", codebook.data_ptr(), codebook.shape[0], index.data_ptr(), index.numel(), ch, _ptr(out),
              *_pargs(pl), row_limit.data_ptr(), index.shape[1], _stream())
    return _result(out, pl, nsplit)


def row_sqnorm(x):
    _chk(x)
    out = torch.empty(x.shape[0], device=x.device, dtype=torch.float32)
    _call("pm_row_sqnorm_f32", x.data_ptr(), x.shape[0], x.shape[1], out.data_ptr(), _stream())
    return out


def pose_compose(face, upper, hands, lower, bs, t, device):
    for ten, dim in ((face, 106), (upper, 78), (hands, 180), (lower, 61)):
        if ten is not None:
            _chk(ten)
            assert ten.is_contiguous() and ten.shape == (bs, t, dim), (ten.shape, dim)
    expression = torch.empty(bs, t, 100, device=device, dtype=torch.float32)
    axis_angle = torch.empty(bs, t, 165, device=device, dtype=torch.float32)
    motion4inf = torch.empty(bs, t, 337, device=device, dtype=torch.float32)
    _call("pm_pose_compose_f32", _ptr(face), _ptr(upper), _ptr(hands), _ptr(lower), expression.data_ptr(),
          axis_angle.data_ptr(), motion4inf.data_ptr(), bs * t, _stream())
    return expression, axis_angle, motion4inf


def global_trans(rec, ref_trans, dt, vel_off=54):
    _chk(rec), _chk(ref_trans)
    assert rec.is_contiguous()
    bs, t, ld = rec.shape
    assert ref_trans.shape == (bs, 3)                      # may be an expanded (stride 0) view of one row
    trans = torch.empty(bs, t, 3, device=rec.device, dtype=torch.float32)
    _call("pm_global_trans_f32", rec.data_ptr(), ld, vel_off, ref_trans.data_ptr(), ref_trans.stride(0), float(dt),
          trans.data_ptr(), bs, t, _stream())
    return trans


# ------------------------------------------------------------------------------------------------------
# tcgen05 tensor-core engine: split-bf16 planes
# ------------------------------------------------------------------------------------------------------


def _round_up(x, m):
    return (x + m - 1) // m * m


class Planes:
    """`nsplit` bf16 planes of a (batch, rows, ch) activation: tensor (nsplit, batch, rows_alloc, ld) bf16
    with x ~ sum_p planes[p].  Only [:, :, :rows, :ch] is meaningful."""
    __slots__ = ("t", "rows", "ch", "slack")

    def __init__(self, t, rows, ch, slack=0):
        self.t, self.rows, self.ch, self.slack = t, rows, ch, slack   # slack: zeroed rows after the last clip

    def flat(self):
        """(nsplit, 1, batch*rows, ld) view: all clips as one tall matrix (needs clip-contiguous rows)."""
        ns, b, r, ld = self.t.shape
        assert self.t.stride(1) == r * self.t.stride(2)
        return Planes(self.t.as_strided((ns, 1, b * r, ld), (self.t.stride(0), b * r * self.t.stride(2), self.t.stride(2), 1),
                                        self.t.storage_offset()), b * r, self.ch, self.slack)

    @property
    def nsplit(self):
        return self.t.shape[0]

    @property
    def batch(self):
        return self.t.shape[1]


def split_bf16(x, nsplit, slack_rows=0):
    """fp32 (batch, rows, ch) view -> Planes (ld = ch rounded up to 8).  `slack_rows` zeroed rows are
    appended after the last clip for strided-view consumers."""
    _chk(x)
    batch, rows, ch = x.shape
    pl = _new_planes(nsplit, (batch, rows), ch, x.device, slack_rows)
    x_bs, ldx = _bs_ld(x)
    _call("pm_split_bf16", x.data_ptr(), x_bs, ldx, batch, rows, ch, pl.t.data_ptr(), pl.t.stride(0), pl.t.stride(1),
          pl.t.stride(2), nsplit | _fmt_bit(pl.t), _stream())
    return pl


class PackedW:
    """Weights of one tap-GEMM for the tensor-core engine: (nsplit, taps, w_rows, ldw) bf16 (or fp16) planes.
    fp16 planes hold W * 2^k with the largest |W| in [16384, 32768) - small weights keep their second plane out of
    the fp16 subnormals - and `acc_scale` = 2^-k / F16_ACT_SCALE is handed to the kernel's epilogue."""
    __slots__ = ("t", "taps", "cout", "cin", "w_rows", "ldw", "acc_scale")

    def __init__(self, w, nsplit):
        """w: fp32 (taps, cout, cin)."""
        taps, cout, cin = w.shape
        bn = 64 if cout <= 64 else 128
        self.taps, self.cout, self.cin = taps, cout, cin
        self.w_rows, self.ldw = _round_up(cout, bn), _round_up(cin, 8)
        full = torch.zeros(taps, self.w_rows, self.ldw, device=w.device, dtype=torch.float32)
        full[:, :cout, :cin] = w
        self.acc_scale = 1.0
        if _PLANE_DTYPE == torch.float16:
            m = float(full.abs().max())
            if m > 0.0 and math.isfinite(m):
                k = math.floor(math.log2(32768.0 / m))
                full = full * (2.0 ** k)
                self.acc_scale = 2.0 ** -k
            self.acc_scale /= F16_ACT_SCALE                  # activation planes arrive pre-scaled (exact power of two)
        planes, rem = [], full
        for _ in range(nsplit):                       # round-to-nearest-even, same as the device split
            p = rem.to(_PLANE_DTYPE)
            planes.append(p)
            rem = rem - p.float()
        self.t = torch.stack(planes).contiguous()


def tapgemm_tc(a: Planes, w: PackedW, bias, *, rows_in=None, rows_out, pad=0, act=ACT_NONE, act_cols=0, slope=0.0,
               residual=None, want_f32=True, out_nsplit=0, out=None, a_view=None, out_slack=0, prefetch=None,
               row_limit=None, rows_per_clip=0):
    """Tensor-core tap-GEMM.  `prefetch`: a tensor (the next GEMM's packed weights) to pull into L2 meanwhile.
    `a_view` = (rows_in, cin, lda) overrides the logical view of the A planes
    (strided convs pass the (rows/s, s*C) view of the same memory).  Returns (fp32 out | None, Planes | None).
    row_limit: optional int32 device tensor of per-clip valid output rows (ragged batch; include/pm_emage.h
    pm_tapgemm_tc_rl); the clip is the batch index, or row // rows_per_clip of a flat (1, clips*rows) launch."""
    t = a.t
    nsplit, batch = t.shape[0], t.shape[1]
    assert nsplit == w.t.shape[0] and t.dtype == w.t.dtype, "A and W must use the same split and plane format"
    fmt = _fmt_bit(t)
    rows_a, cin, lda = (a.rows, a.ch, t.stride(2)) if a_view is None else a_view
    if rows_in is not None:
        rows_a = rows_in
    assert cin == w.cin, (cin, w.cin)
    cout = w.cout
    dev = t.device
    out_f = None
    if want_f32:
        out_f = out if out is not None else torch.empty(batch, rows_out, cout, device=dev, dtype=torch.float32)
        assert out_f.shape == (batch, rows_out, cout)
    o_bs, ldo = _bs_ld(out_f) if out_f is not None else (0, 0)
    out_p = None
    if out_nsplit:
        out_p = _new_planes(out_nsplit, (batch, rows_out), cout, dev, out_slack, dtype=t.dtype)
    r_bs, ldr = _bs_ld(residual) if residual is not None else (0, 0)
    if residual is not None:
        _chk(residual)
        assert residual.shape == (batch, rows_out, cout)
    ob = (None, 0, 0, 0) if out_p is None else (out_p.t.data_ptr(), out_p.t.stride(0), out_p.t.stride(1), out_p.t.stride(2))
    pf_ptr, pf_bytes = (None, 0) if prefetch is None else (prefetch.data_ptr(), prefetch.numel() * prefetch.element_size())
    if row_limit is None:
        _call("pm_tapgemm_tc", t.data_ptr(), t.stride(0), t.stride(1), lda, batch, rows_a, cin,
              w.t.data_ptr(), w.t.stride(0), w.w_rows, w.ldw, w.taps, pad, nsplit | fmt,
              _ptr(bias), rows_out, cout, _ptr(residual), r_bs, ldr, act, act_cols, float(slope), float(w.acc_scale),
              _ptr(out_f), o_bs, ldo, ob[0], ob[1], ob[2], ob[3], out_nsplit | (fmt if out_nsplit else 0),
              pf_ptr, pf_bytes, _stream())
    else:
        _chk_limit(row_limit, -(-batch * rows_out // rows_per_clip) if rows_per_clip else batch)
        _call("pm_tapgemm_tc_rl", t.data_ptr(), t.stride(0), t.stride(1), lda, batch, rows_a, cin,
              w.t.data_ptr(), w.t.stride(0), w.w_rows, w.ldw, w.taps, pad, nsplit | fmt,
              _ptr(bias), rows_out, cout, _ptr(residual), r_bs, ldr, act, act_cols, float(slope), float(w.acc_scale),
              _ptr(out_f), o_bs, ldo, ob[0], ob[1], ob[2], ob[3], out_nsplit | (fmt if out_nsplit else 0),
              pf_ptr, pf_bytes, row_limit.data_ptr(), rows_per_clip, _stream())
    return out_f, out_p


# ------------------------------------------------------------------------------------------------------
# CaMN / DisCo
# ------------------------------------------------------------------------------------------------------


def lstm_bidir(xproj, whh, barrier, hidden):
    """One bidirectional LSTM layer.  xproj (batch, t, 8*hidden) = W_ih x + b for [forward | backward] (gates
    i,f,g,o), whh (2, 4*hidden, hidden).  Returns (batch, t, 2*hidden) = [forward h | backward h]."""
    _chk(xproj), _chk(whh)
    assert xproj.is_contiguous() and whh.is_contiguous() and whh.shape == (2, 4 * hidden, hidden)
    batch, t, w = xproj.shape
    assert w == 8 * hidden
    y = torch.empty(batch, t, 2 * hidden, device=xproj.device, dtype=torch.float32)
    _call("pm_lstm_bidir_f32", xproj.data_ptr(), xproj.stride(0), xproj.stride(1), whh.data_ptr(), y.data_ptr(),
          y.stride(0), y.stride(1), barrier.data_ptr(), batch, t, hidden, _stream())
    return y


def rot6d_to_aa(rot6d, slot, n_sel):
    """rot6d (..., n_sel*6) -> axis-angle (..., 165); slot: int32[55] device tensor (position among the selected
    joints or -1)."""
    _chk(rot6d)
    assert rot6d.is_contiguous() and rot6d.shape[-1] == n_sel * 6
    rows = rot6d.numel() // (n_sel * 6)
    out = torch.empty(*rot6d.shape[:-1], 165, device=rot6d.device, dtype=torch.float32)
    _call("pm_rot6d_to_aa_f32", rot6d.data_ptr(), rows, n_sel, slot.data_ptr(), out.data_ptr(), _stream())
    return out


def softmax2_mix(sel, c1, c2, out=None):
    """out[..., :] = softmax(sel[..., 0:2])[0] * c1 + [1] * c2 (out may be a column slice of a wider tensor)."""
    _chk(sel), _chk(c1), _chk(c2)
    assert sel.is_contiguous() and c1.is_contiguous() and c2.is_contiguous() and sel.shape[-1] == 2
    ch = c1.shape[-1]
    rows = c1.numel() // ch
    if out is None:
        out = torch.empty_like(c1)
    _call("pm_softmax2_mix_f32", sel.data_ptr(), c1.data_ptr(), c2.data_ptr(), out.data_ptr(), rows, ch, out.stride(-2), _stream())
    return out
