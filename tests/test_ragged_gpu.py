"""Ragged batches on the GPU: every `_rl` entry point against float64 torch and against its plain twin run on each clip
alone, and generate_ragged() / RaggedPipeline against per-clip generate() and the committed goldens."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle.weights import synth_audio
from helpers import build_product

pytestmark = pytest.mark.gpu
PARTS = ("face", "upper", "hands", "lower")


@pytest.fixture(scope="module")
def product():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return build_product(seed=0)


@pytest.fixture(autouse=True)
def _restore_precision():
    from pantomatrix_b200.emage_audio import engine
    yield
    engine.set_precision(engine.DEFAULT_PRECISION)


def _i32(v):
    return torch.tensor(v, dtype=torch.int32, device="cuda")


def _ragged(lens, rows, ch, g):
    """(clips, rows, ch) activations, zero beyond each clip's length (the layout the `_rl` kernels keep)."""
    x = torch.randn(len(lens), rows, ch, generator=g).cuda()
    for b, n in enumerate(lens):
        x[b, n:] = 0
    return x


# (taps, stride, pad, cin, cout, rows): the WavEncoder's k=15 / pad 7 conv (halo mode, two CTAs per SM), the VQ k=3
# conv (CTA pairs in fp16x3), a stride-6 conv (strided (rows/s, s*C) view) and a Linear (one tall matrix)
CONVS = [(15, 1, 7, 64, 64, 700), (3, 1, 1, 256, 256, 512), (15, 6, 0, 64, 64, 600), (1, 1, 0, 768, 768, 64)]


@pytest.mark.parametrize("precision", ["fp32", "bf16x6", "fp16x3"])
@pytest.mark.parametrize("shape", CONVS, ids=["k15", "k3", "stride6", "linear"])
def test_tapgemm_rl_matches_each_clip_alone(product, precision, shape):
    from pantomatrix_b200.emage_audio import engine as E
    E.set_precision(precision)
    taps, stride, pad, cin, cout, rows = shape
    g = torch.Generator().manual_seed(taps * 7 + stride)
    w, b = torch.randn(taps, cout, cin, generator=g) / (taps * cin) ** 0.5, torch.randn(cout, generator=g) * 0.1
    conv = E._Conv(w.cuda().contiguous(), b.cuda(), stride, pad)
    lens_in = [rows, rows // 3, 17, 0, rows - 5, 40] if taps > 1 else [64, 11, 0, 63, 64, 1]
    out_len = lambda n: max(0, (n + 2 * pad - taps) // stride + 1) if n else 0
    x = _ragged(lens_in, rows, cin, g)
    lim = _i32([out_len(n) for n in lens_in])
    got = conv(x, want="fp" if precision != "fp32" else "f", row_limit=lim)
    gf = got.f if isinstance(got, E.ops.Act) else got
    want64 = F.conv1d(x.double().transpose(1, 2), w.double().permute(1, 2, 0).cuda(), b.double().cuda(),
                      stride=stride, padding=pad).transpose(1, 2)
    for c, n in enumerate(lens_in):
        m = out_len(n)
        assert (gf[c, m:] == 0).all(), (c, m)                                        # rows beyond the limit: exact 0
        if precision != "fp32":
            pl = got.p.t[:, c, m:, :cout]
            assert (pl == 0).all(), c
        if m == 0:
            continue
        alone = conv(x[c:c + 1, :n].contiguous())                                    # the plain twin on the clip alone
        assert torch.equal(gf[c, :m], alone[0, :m]), (c, (gf[c, :m] - alone[0, :m]).abs().max())
        err = (gf[c, :m].double() - want64[c, :m]).abs().max().item()
        assert err < 1e-4, (c, err)


@pytest.mark.parametrize("precision", ["fp32", "fp16x3"])
def test_attention_rl_matches_each_clip_alone(product, precision):
    from pantomatrix_b200 import ops
    from pantomatrix_b200.emage_audio import engine as E
    E.set_precision(precision)
    g = torch.Generator().manual_seed(5)
    q_len, k_len = [64, 11, 40, 7, 64], [64, 12, 40, 0, 63]          # includes k_len = q_len + 1 and k_len = 0
    B, H, hd = len(q_len), 4, 192
    E_ = H * hd
    q, k, v = (torch.randn(B, 64, E_, generator=g).cuda() * 0.5 for _ in range(3))
    ql, kl = _i32(q_len), _i32(k_len)

    def run(qq, kk, vv, bs, tq, tk, **lim):
        if precision == "fp32":
            return ops.attention(qq.reshape(bs * tq, E_), kk.reshape(bs * tk, E_), vv.reshape(bs * tk, E_), bs, H, tq, tk,
                                 hd, nsplit=0, f32=True, **lim).view(bs, tq, E_)
        pl = lambda t: ops.split_bf16(t.contiguous(), 2)
        return ops.attention_tc(pl(qq), 0, pl(kk), 0, pl(vv), 0, bs, H, tq, tk, hd, nsplit=0, f32=True, **lim).view(bs, tq, E_)

    got = run(q, k, v, B, 64, 64, q_len=ql, k_len=kl)
    for c in range(B):
        tq, tk = q_len[c], k_len[c]
        assert (got[c, tq:] == 0).all()
        if tk == 0:
            assert (got[c] == 0).all()
            continue
        alone = run(q[c:c + 1, :tq], k[c:c + 1, :tk], v[c:c + 1, :tk], 1, tq, tk)
        assert torch.equal(got[c, :tq], alone[0]), (c, (got[c, :tq] - alone[0]).abs().max())
        ref = torch.softmax(q[c, :tq].double().view(tq, H, hd).transpose(0, 1) @
                            k[c, :tk].double().view(tk, H, hd).permute(1, 2, 0) / hd ** 0.5, -1) @ \
            v[c, :tk].double().view(tk, H, hd).transpose(0, 1)
        assert (got[c, :tq].double() - ref.transpose(0, 1).reshape(tq, E_)).abs().max() < 1e-4


@pytest.mark.parametrize("precision", ["fp32", "fp16x3"])
def test_wav_stem_rl_reads_zero_beyond_each_slice(product, precision):
    from pantomatrix_b200 import ops
    from pantomatrix_b200.emage_audio import engine as E
    E.set_precision(precision)
    model, _ = product
    w1, b1, wd, bd, stride, pad = model._eng().wav_face.stem
    g = torch.Generator().manual_seed(9)
    n, windows, bs = 64 * 533, 2, 3
    audio = torch.randn(bs, 3 * n, generator=g).cuda() * 0.1                     # non-zero audio after every slice
    nv = [[n, 11 * 533, 0], [40 * 533, n, 5863]]                                 # window-major (w, b)
    ns = 2 if precision == "fp16x3" else 0
    y, sc = ops.wav_stem(audio, 3 * n, n, bs, windows, n, w1, b1, wd, bd, stride=stride, pad=pad, slope=0.01, nsplit=ns,
                         n_valid=_i32(sum(nv, [])))
    for w in range(windows):
        for b in range(bs):
            s, cnt = w * n, nv[w][b]
            rows = (cnt + 2 * pad - 15) // stride + 1 if cnt else 0
            assert (sc[w * bs + b, rows:] == 0).all()
            if not cnt:
                continue
            ya, sa = ops.wav_stem(audio[b:b + 1, s:s + cnt].contiguous(), cnt, 0, 1, 1, cnt, w1, b1, wd, bd, stride=stride,
                                  pad=pad, slope=0.01, nsplit=ns)
            assert torch.equal(sc[w * bs + b, :rows], sa[0]), (w, b)
            if ns:
                C = w1.shape[0]
                assert torch.equal(y.t[:, w * bs + b, :rows, :C], ya.t[:, 0, :, :C]) and (y.t[:, w * bs + b, rows:, :C] == 0).all()
            else:
                assert torch.equal(y[w * bs + b, :rows], ya[0]) and (y[w * bs + b, rows:] == 0).all()


def test_window_input_and_gather_rows_rl(product):
    from pantomatrix_b200 import ops
    model, vqm = product
    emb = model._eng().mask_embedding
    seed = torch.randn(3, 4, 337).cuda()
    lim = _i32([64, 9, 0])
    x = ops.window_input(None, None, seed, emb, 60, 64, 4, shape=(3, 200, 337), row_limit=lim)
    ref = ops.window_input(None, None, seed, emb, 60, 64, 4, shape=(3, 200, 337))
    for b, n in enumerate([64, 9, 0]):
        assert torch.equal(x[b, :n], ref[b, :n]) and (x[b, n:] == 0).all()
    cb = vqm.engine().codebook["upper"]
    idx = torch.randint(0, 256, (3, 50), device="cuda")
    lim = _i32([50, 7, 0])
    y = ops.gather_rows(cb, idx, row_limit=lim)
    for b, n in enumerate([50, 7, 0]):
        assert torch.equal(y[b, :n], cb[idx[b, :n]]) and (y[b, n:] == 0).all()


# ---- end to end --------------------------------------------------------------------------------------------------


def _per_clip(model, vqm, audios):
    from pantomatrix_b200.pipeline import generate
    return [generate(model, vqm, a[None]) for a in audios]


def _lengths(seed, n):
    rng = np.random.default_rng(seed)
    # every plan shape: no tail (124 frames), a tail of T <= 25 rows (131), a single window (40), a full-length spill
    # (64 + 60k frames + a tail of 61..63 rows: 186), then random 1-12 s clips
    frames = [124, 131, 40, 186] + list(rng.integers(30, 360, n - 4))
    return [-(-int(f) * 16000 // 30) + int(rng.integers(0, 500)) for f in frames]


def test_ragged_fp32_is_bit_identical_to_each_clip_alone(product):
    from pantomatrix_b200.emage_audio import engine as E
    from pantomatrix_b200.pipeline import generate_ragged
    E.set_precision("fp32")
    model, vqm = product
    audios = [torch.from_numpy(synth_audio(1, n, 100 + i))[0].cuda() for i, n in enumerate(_lengths(0, 16))]
    got = generate_ragged(model, vqm, audios)
    for i, (lat, pred) in enumerate(_per_clip(model, vqm, audios)):
        for k in lat:
            assert torch.equal(got[i][0][k], lat[k]), (i, k, (got[i][0][k] - lat[k]).abs().max())
        for k in pred:
            assert torch.equal(got[i][1][k], pred[k]), (i, k, (got[i][1][k] - pred[k]).abs().max())


def test_ragged_fp16x3_is_bit_identical_to_each_clip_alone(product):
    from pantomatrix_b200.emage_audio import engine as E
    from pantomatrix_b200.pipeline import generate_ragged
    E.set_precision("fp16x3")
    model, vqm = product
    audios = [torch.from_numpy(synth_audio(1, n, 200 + i))[0].cuda() for i, n in enumerate(_lengths(1, 16))]
    got = generate_ragged(model, vqm, audios)
    for i, (lat, pred) in enumerate(_per_clip(model, vqm, audios)):
        for k, v in list(lat.items()) + list(pred.items()):
            other = got[i][0][k] if k in lat else got[i][1][k]
            assert torch.equal(other, v), (i, k, (other - v).abs().max().item())


# Clips whose audio runs past the batch's last window: no tail (remain == 0: 64 and 124 frames), a dropped tail
# (remain <= pre: 126 frames) and a 63-row tail whose sample count has a large fraction of a frame (123 frames).
EDGE_BATCHES = [[34134], [67200], [66100], [66134], [66134, 21600], [67200, 66100, 21600]]


@pytest.mark.parametrize("precision", ["fp32", "fp16x3"])
@pytest.mark.parametrize("lens", EDGE_BATCHES, ids=["no_tail64", "drop_tail126", "tail63", "no_tail124",
                                                    "drop_tail_short40", "mixed"])
def test_ragged_clips_longer_than_their_windows(product, precision, lens):
    from pantomatrix_b200.emage_audio import engine as E
    from pantomatrix_b200.pipeline import generate_ragged
    E.set_precision(precision)
    model, vqm = product
    audios = [torch.from_numpy(synth_audio(1, n, 400 + i))[0].cuda() for i, n in enumerate(lens)]
    got = generate_ragged(model, vqm, audios)
    for i, (lat, pred) in enumerate(_per_clip(model, vqm, audios)):
        for k, v in list(lat.items()) + list(pred.items()):
            other = got[i][0][k] if k in lat else got[i][1][k]
            assert torch.equal(other, v), (i, k)


@pytest.mark.parametrize("precision", ["fp32", "bf16x6", "fp16x3"])
@pytest.mark.parametrize("cases", [("tail11", "clip10s", "drop_tail", "short40"), ("drop_tail", "short40")],
                         ids=["all", "drop_tail_short40"])
def test_ragged_goldens(product, golden_dir, precision, cases):
    """Golden clips (tail11 x2, clip10s, drop_tail x2, short40 x2, or drop_tail + short40 alone) in one ragged batch:
    every clip meets the gates test_emage_gpu.py applies to its golden - indices exact, latents and logits close,
    SMPL-X outputs within 1e-3 of the reference's."""
    from pantomatrix_b200.emage_audio import engine as E
    from pantomatrix_b200.pipeline import generate_ragged
    from test_emage_gpu import _pose_checks
    E.set_precision(precision)
    model, vqm = product
    audios, gold = [], []
    for case in cases:
        g = np.load(os.path.join(golden_dir, f"case_{case}.npz"))
        a = torch.from_numpy(synth_audio(int(g["bs"]), int(g["n_samples"]), int(g["audio_seed"]))).cuda()
        for b in range(a.shape[0]):
            audios.append(a[b])
            gold.append((case, g, b))
    got = generate_ragged(model, vqm, audios)
    for (case, g, b), (lat, pred) in zip(gold, got):
        tag = f"{case}[{b}] {precision}"
        for p in PARTS:
            assert lat["cls_" + p].shape[1] == g["idx_cls_" + p].shape[1], (tag, "emitted length")
            idx = lat["cls_" + p].argmax(-1)[0].cpu().numpy()
            assert np.array_equal(idx, g["idx_cls_" + p][b]), (tag, p, int((idx != g["idx_cls_" + p][b]).sum()))
            np.testing.assert_allclose(lat["rec_" + p][0].cpu().numpy()[::7], g["rec_" + p][b], atol=1e-3, rtol=0)
            np.testing.assert_allclose(lat["cls_" + p][0].cpu().numpy()[::7], g["cls_" + p][b], atol=2e-3, rtol=0)
        face_idx = vqm.vq_model_face._index_of(lat["rec_face"]).cpu().numpy()
        assert np.array_equal(face_idx[0], g["idx_l2_face"][b]), tag
        one = lambda k: torch.from_numpy(g[k][b:b + 1])
        _pose_checks(pred, one("motion_axis_angle"), one("expression"), one("trans"), tag)
        assert (pred["all_motion4inference"].cpu() - one("all_motion4inference")).abs().max() < 1e-3, tag


def test_ragged_pipeline_replays_equal_eager(product):
    from pantomatrix_b200.emage_audio import engine as E
    from pantomatrix_b200.pipeline import RaggedPipeline, generate_ragged
    E.set_precision("fp32")
    model, vqm = product
    pipe = RaggedPipeline(model, vqm, batch=4, max_samples=200000, warmup=1)
    for seed, lens in ((3, [70000, 21600, 160000]), (4, [66134, 200000, 40000, 30000])):
        audios = [torch.from_numpy(synth_audio(1, n, seed * 10 + i))[0].cuda() for i, n in enumerate(lens)]
        got = pipe(audios)
        want = generate_ragged(model, vqm, audios)
        assert len(got) == len(lens)
        for (gl, gp), (wl, wp) in zip(got, want):
            for k in wl:
                assert torch.equal(gl[k], wl[k]), k
            for k in wp:
                assert torch.equal(gp[k], wp[k]), k
    # a capacity whose longest clip has no tail window: its audio runs past the last window
    edge = RaggedPipeline(model, vqm, batch=2, max_samples=66134, warmup=1)
    for lens in ([66134], [66100, 21600]):
        audios = [torch.from_numpy(synth_audio(1, n, 500 + i))[0].cuda() for i, n in enumerate(lens)]
        for (gl, gp), (wl, wp) in zip(edge(audios), generate_ragged(model, vqm, audios)):
            for k in wl:
                assert torch.equal(gl[k], wl[k]), k
            for k in wp:
                assert torch.equal(gp[k], wp[k]), k
    with pytest.raises(ValueError):
        pipe([torch.zeros(1000, device="cuda")] * 5)
    with pytest.raises(ValueError):
        pipe([torch.zeros(200001, device="cuda")])


def test_demo_batch_writes_the_same_files_as_one_at_a_time(tmp_path):
    """examples/emage_audio_demo.py --batch 4 (ragged groups of sorted files) == --batch 1, fp32 engine."""
    import subprocess
    import sys
    import wave
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    wavs = tmp_path / "wavs"
    wavs.mkdir()
    for i, n in enumerate([70000, 21600, 160000, 66134, 45000, 98000]):
        pcm = (synth_audio(1, n, 300 + i)[0] * 20000).clip(-32768, 32767).astype(np.int16)
        with wave.open(str(wavs / f"clip{i}.wav"), "wb") as w:
            w.setnchannels(1), w.setsampwidth(2), w.setframerate(16000), w.writeframes(pcm.tobytes())
    env = dict(os.environ, PM_EMAGE_PRECISION="fp32")
    outs = {}
    for batch in (1, 4):
        out = tmp_path / f"out{batch}"
        subprocess.run([sys.executable, os.path.join(root, "examples", "emage_audio_demo.py"), "--synthetic",
                        "--audio_folder", str(wavs), "--save_folder", str(out), "--batch", str(batch)],
                       check=True, env=env, cwd=str(tmp_path))
        outs[batch] = out
    names = sorted(os.listdir(outs[1]))
    assert names == sorted(os.listdir(outs[4])) and len(names) == 6
    for name in names:
        a, b = np.load(outs[1] / name), np.load(outs[4] / name)
        assert sorted(a.files) == sorted(b.files)
        for k in a.files:
            assert np.array_equal(a[k], b[k]), (name, k)
