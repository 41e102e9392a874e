"""Ragged batches without a GPU: the per-clip geometry of engine.RaggedPlan against the per-clip arithmetic it is
derived from, and generate_ragged() against per-clip generate() with every kernel replaced by tests/fake_ops.py plus
limit-aware stand-ins of the `_rl` entry points (include/pm_emage.h) defined here."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import fake_ops
from oracle.weights import synth_audio

PARTS = ("face", "upper", "hands", "lower")
SPF = 16000 // 30


def _samples(frames):
    """The smallest sample count inference() turns into `frames` frames (M.py:345)."""
    return -(-frames * 16000 // 30)


# ---- limit-aware stand-ins ---------------------------------------------------------------------------------------


def _limit_rows(y, row_limit, prev=None):
    """y (clips, rows, ch): rows >= row_limit[clip] -> 0; a negative limit keeps `prev` (the rows are not written)."""
    lim = row_limit.cpu().long()
    r = torch.arange(y.shape[1])[None, :, None]
    y = torch.where(r >= lim[:y.shape[0], None, None], torch.zeros((), dtype=y.dtype), y)
    if prev is not None:
        y = torch.where(lim[:y.shape[0], None, None] < 0, prev, y)
    return y


def tapgemm(a, w, bias, *, row_limit=None, out=None, **kw):
    y = fake_ops.tapgemm(a, w, bias, **kw)
    if row_limit is not None:
        y = _limit_rows(y, row_limit, None if out is None else out.clone())
    if out is not None:
        out.copy_(y)
        return out
    return y


def tapgemm_tc(a, w, bias, *, row_limit=None, rows_per_clip=0, want_f32=True, out_nsplit=0, out=None, out_slack=0,
               residual=None, **kw):
    if row_limit is None:
        return fake_ops.tapgemm_tc(a, w, bias, want_f32=want_f32, out_nsplit=out_nsplit, out=out, out_slack=out_slack,
                                   residual=residual, **kw)
    y, _ = fake_ops.tapgemm_tc(a, w, bias, want_f32=True, residual=residual, **kw)
    batch, rows, cout = y.shape
    shape = (batch * rows // rows_per_clip, rows_per_clip, cout) if rows_per_clip else y.shape
    prev = out.reshape(shape).clone() if out is not None else torch.zeros(shape)
    y = _limit_rows(y.reshape(shape), row_limit, prev).reshape(batch, rows, cout)
    pl = fake_ops._mk_planes(y, out_nsplit, out_slack) if out_nsplit else None
    if not want_f32:
        return None, pl
    if out is not None:
        out.copy_(y)
        return out, pl
    return y.contiguous(), pl


def wav_stem(audio, a_bs, a_ws, batch, windows, n_samples, w1, b1, wd, bd, *, stride, pad, slope, offset=0, nsplit=0,
             n_valid=None):
    if n_valid is None:
        return fake_ops.wav_stem(audio, a_bs, a_ws, batch, windows, n_samples, w1, b1, wd, bd, stride=stride, pad=pad,
                                 slope=slope, offset=offset, nsplit=nsplit)
    flat = audio.reshape(-1)
    nv = n_valid.cpu().long()
    seqs = torch.stack([flat[offset + b * a_bs + w * a_ws: offset + b * a_bs + w * a_ws + n_samples]
                        for w in range(windows) for b in range(batch)])
    seqs = torch.where(torch.arange(n_samples)[None] < nv[:, None], seqs, torch.zeros(()))   # zero padding beyond
    x = seqs.unsqueeze(1)
    y1 = F.leaky_relu(F.conv1d(x, w1.unsqueeze(1), b1, stride=stride, padding=pad), slope).transpose(1, 2)
    sc = F.conv1d(x, wd.unsqueeze(1), bd, stride=stride, padding=pad).transpose(1, 2)
    rows = torch.where(nv > 0, (nv + 2 * pad - w1.shape[1]) // stride + 1, torch.zeros_like(nv))
    y1, sc = _limit_rows(y1, rows).contiguous(), _limit_rows(sc, rows).contiguous()
    return (fake_ops._mk_planes(y1, nsplit) if nsplit else y1), sc


def attention(q, k, v, batch, heads, tq, tk, head_dim, nsplit=0, f32=True, q_len=None, k_len=None):
    if k_len is None:
        return fake_ops.attention(q, k, v, batch, heads, tq, tk, head_dim, nsplit=nsplit, f32=f32)
    E = heads * head_dim
    qq = q[:, :E].reshape(batch, tq, heads, head_dim).transpose(1, 2)
    kk = k[:, :E].reshape(batch, tk, heads, head_dim).transpose(1, 2)
    vv = v[:, :E].reshape(batch, tk, heads, head_dim).transpose(1, 2)
    ql, kl = q_len.cpu().long()[:batch], k_len.cpu().long()[:batch]
    s = qq @ kk.transpose(-1, -2) / head_dim ** 0.5
    keep = torch.arange(tk)[None, :] < kl[:, None]                               # (batch, tk)
    s = s.masked_fill(~keep[:, None, None, :], float("-inf"))
    p = torch.nan_to_num(torch.softmax(s, -1), nan=0.0)                          # k_len = 0: zeros, never 0/0
    o = (p @ (vv * keep[:, None, :, None])).transpose(1, 2).reshape(batch, tq, E)
    o = _limit_rows(o, torch.where(kl > 0, ql, torch.zeros_like(ql)))
    return fake_ops._res(o.reshape(batch * tq, E), nsplit, f32, lead=(batch, tq))


def attention_tc(q, q_col0, k, k_col0, v, v_col0, batch, heads, tq, tk, head_dim, nsplit=2, f32=False, q_len=None,
                 k_len=None):
    E = heads * head_dim
    val = lambda pl, c0, rows: (pl.t[:, :, :rows, c0:c0 + E].float().sum(0) / 64.0).reshape(batch * rows, E)
    return attention(val(q, q_col0, tq), val(k, k_col0, tk), val(v, v_col0, tk), batch, heads, tq, tk, head_dim,
                     nsplit=nsplit, f32=f32, q_len=q_len, k_len=k_len)


def window_input(motion, mask, seed, mask_embedding, start, win_len, pre, nsplit=0, f32=True, shape=None, row_limit=None):
    y = fake_ops.window_input(motion, mask, seed, mask_embedding, start, win_len, pre, nsplit=0, shape=shape)
    if row_limit is not None:
        y = _limit_rows(y, row_limit)
    return fake_ops._res(y.contiguous(), nsplit, f32)


def gather_rows(codebook, index, nsplit=0, f32=True, row_limit=None):
    if row_limit is None:
        return fake_ops.gather_rows(codebook, index, nsplit=nsplit, f32=f32)
    y = _limit_rows(codebook[index], row_limit)
    return fake_ops._res(y, nsplit, f32, lead=(index.shape[0], index.shape[1]))


RAGGED_FAKES = dict(tapgemm=tapgemm, tapgemm_tc=tapgemm_tc, wav_stem=wav_stem, attention=attention,
                    attention_tc=attention_tc, window_input=window_input, gather_rows=gather_rows)


@pytest.fixture()
def cpu_product(monkeypatch):
    import pantomatrix_b200.ops as real
    from helpers import build_product
    from pantomatrix_b200.emage_audio import engine, modeling
    for name in dir(fake_ops):
        if not name.startswith("_") and callable(getattr(fake_ops, name)) and hasattr(real, name):
            monkeypatch.setattr(real, name, getattr(fake_ops, name))
    for name, fn in RAGGED_FAKES.items():
        monkeypatch.setattr(real, name, fn)
    monkeypatch.setattr(modeling, "_require_cuda", lambda module, what: torch.device("cpu"))
    monkeypatch.setitem(engine._STATE, "nsplit", 0)
    monkeypatch.setitem(engine._STATE, "precision", "fp32")
    monkeypatch.setattr(real, "_PLANE_DTYPE", real._PLANE_DTYPE)
    return build_product(seed=0, device="cpu")


# ---- the plan ----------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("golden", [False, True])
def test_plan_tables_match_per_clip_arithmetic(golden):
    from pantomatrix_b200.emage_audio.engine import RaggedPlan, wav_block_lens, wav_out_len, window_plan
    ns = [70000, 66134, 21600, 160000] if golden else [_samples(f) for f in range(5, 701)]
    ok = [n for n in ns if window_plan(n * 30 // 16000, 64, 4) and window_plan(n * 30 // 16000, 64, 4)[0][0] >= 0]
    for n in ns:
        if n not in ok:
            with pytest.raises(RuntimeError):
                RaggedPlan([n], 64, 4)
    plan = RaggedPlan(ok, 64, 4, batch=len(ok) + 1)
    assert plan.batch == len(ok) + 1 and plan.windows == max(len(window_plan(n * 30 // 16000, 64, 4)) for n in ok)
    for b, n in enumerate(ok):
        wp = window_plan(n * 30 // 16000, 64, 4)
        rows = [e - s for s, e, _ in wp] + [0] * (plan.windows - len(wp))
        assert list(plan.win_rows[:, b]) == rows
        assert list(plan.n_valid[:, b]) == [r * SPF for r in rows]
        assert list(plan.dest_rows[:, b]) == [r if r else -1 for r in rows]
        assert plan.out_len[b] == sum(k for _, _, k in wp)
        for j, r in enumerate(rows):
            assert list(plan.wav_rows[:, j, b]) == (wav_block_lens(r * SPF) if r else [0] * 6)
            assert plan.body_keys[j, b] == (wav_out_len(r * SPF) if r else 0)
            if 0 < r <= 25:
                assert plan.body_keys[j, b] == r + 1                # M.py:278-281: the body stream is not truncated
    assert not plan.win_rows[:, -1].any() and plan.out_len[-1] == 0   # unused slot: no windows
    assert plan.capacity_frames >= plan.out_len.max()
    with pytest.raises(ValueError):
        RaggedPlan(ok[:3], 64, 4, batch=2)


def test_tail11_has_one_more_body_key_than_rows():
    from pantomatrix_b200.emage_audio.engine import RaggedPlan
    plan = RaggedPlan([70000], 64, 4)
    assert list(plan.win_rows[:, 0]) == [64, 64, 11] and list(plan.body_keys[:, 0]) == [64, 64, 12]


# ---- the fakes honour the contract -------------------------------------------------------------------------------


def test_fakes_zero_padded_rows_and_mask_keys():
    g = torch.Generator().manual_seed(0)
    lim = torch.tensor([3, 0, 5, -1], dtype=torch.int32)
    prev = torch.full((4, 6, 8), 7.0)
    y = tapgemm(torch.randn(4, 6, 5, generator=g), torch.randn(3, 8, 5, generator=g), torch.randn(8, generator=g),
                pad=1, row_limit=lim, out=prev)
    assert (y[0, 3:] == 0).all() and (y[1] == 0).all() and (y[2, 5:] == 0).all() and (y[3] == 7).all()
    assert (y[0, :3] != 0).all()
    q = torch.randn(2 * 5, 4 * 192, generator=g)
    kv = torch.randn(2 * 6, 4 * 192, generator=g)
    ql, kl = torch.tensor([4, 5], dtype=torch.int32), torch.tensor([5, 0], dtype=torch.int32)
    o = attention(q, kv, kv, 2, 4, 5, 6, 192, q_len=ql, k_len=kl).view(2, 5, -1)
    ref = fake_ops.attention(q[:4], kv[:5], kv[:5], 1, 4, 4, 5, 192).view(1, 4, -1)
    assert torch.allclose(o[0, :4], ref[0], atol=1e-6) and (o[0, 4:] == 0).all() and (o[1] == 0).all()


# ---- end to end on the fakes -------------------------------------------------------------------------------------


def test_generate_ragged_reproduces_per_clip_generate(cpu_product):
    from pantomatrix_b200.pipeline import generate, generate_ragged
    model, vqm = cpu_product
    ns = [70000, 21600, 66134]                         # tail of 11 rows, a single 40-row window, no tail
    audios = [torch.from_numpy(synth_audio(1, n, 11 + i))[0] for i, n in enumerate(ns)]
    spk = [0, 0, 0]                                   # the synthetic checkpoint has one speaker
    got = generate_ragged(model, vqm, audios, speaker_ids=spk)
    assert len(got) == len(ns)
    for i, a in enumerate(audios):
        lat, pred = generate(model, vqm, a[None], torch.tensor([[spk[i]]]))
        glat, gpred = got[i]
        assert set(glat) == set(lat) and set(gpred) == set(pred)
        for k in lat:
            assert glat[k].shape == lat[k].shape, k
            # CPU convolutions round differently per batch shape: ~5e-5 after the stack; a padded row read as data
            # would be O(0.1).  (On the GPU the fp32 engine is checked bit for bit, tests/test_ragged_gpu.py.)
            np.testing.assert_allclose(glat[k].numpy(), lat[k].numpy(), atol=5e-4, rtol=0, err_msg=k)
        for p in PARTS:
            assert torch.equal(glat["cls_" + p].argmax(-1), lat["cls_" + p].argmax(-1)), p
        for k in pred:
            assert gpred[k].shape == pred[k].shape, k
            np.testing.assert_allclose(gpred[k].numpy(), pred[k].numpy(), atol=1e-3, rtol=0, err_msg=k)


@pytest.mark.parametrize("lens", [[34134], [67200], [66100], [66134, 21600]],
                         ids=["no_tail64", "drop_tail126", "tail63", "drop_tail_short40"])
def test_generate_ragged_clips_longer_than_their_windows(cpu_product, lens):
    """Clips whose audio runs past the batch's last window (no tail, a dropped tail, a 63-row tail with a large
    fraction of a frame left over) as the longest clip of their batch: only the samples the windows read are staged."""
    from pantomatrix_b200.emage_audio.engine import RaggedPlan
    from pantomatrix_b200.pipeline import generate, generate_ragged
    model, vqm = cpu_product
    assert max(lens) > RaggedPlan(lens, 64, 4).capacity_samples
    audios = [torch.from_numpy(synth_audio(1, n, 21 + i))[0] for i, n in enumerate(lens)]
    got = generate_ragged(model, vqm, audios)
    for i, a in enumerate(audios):
        lat, pred = generate(model, vqm, a[None])
        for k in lat:
            np.testing.assert_allclose(got[i][0][k].numpy(), lat[k].numpy(), atol=5e-4, rtol=0, err_msg=k)
        for p in PARTS:
            assert torch.equal(got[i][0]["cls_" + p].argmax(-1), lat["cls_" + p].argmax(-1)), p
        for k in pred:
            np.testing.assert_allclose(got[i][1][k].numpy(), pred[k].numpy(), atol=1e-3, rtol=0, err_msg=k)


def test_generate_ragged_rejects_masked_motion_and_short_clips(cpu_product):
    from pantomatrix_b200.pipeline import generate_ragged
    model, vqm = cpu_product
    with pytest.raises(ValueError):
        generate_ragged(model, vqm, [torch.zeros(21600)], masked_motion=torch.zeros(1, 40, 337))
    with pytest.raises(RuntimeError):
        generate_ragged(model, vqm, [torch.zeros(21600), torch.zeros(1000)])
