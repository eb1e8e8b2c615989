"""CPU tests of the oracle: golden vectors made from the reference's own plumbing, and independent
re-implementations of the two big graphs (torch.stft + torchaudio filterbank; torch conv2d)."""
import numpy as np
import pytest
import torch

from oracle import mel, embedding, heads, streaming
from helpers import emb_weights, head, class_mapping, golden_cases, load_case


@pytest.mark.parametrize("tag", golden_cases("predict_clip"))
def test_state_machine_matches_reference_plumbing(tag):
    c = load_case(tag)
    hs = {n: head(n) for n in c["names"]}
    om = streaming.OracleModel(emb_weights(int(c["emb_seed"])), hs, class_mapping(c["names"]),
                               feature_init=c["feature_init"])
    res = om.predict_clip(c["pcm"], padding=int(c["padding"]), chunk_size=int(c["chunk"]), **c["kw"])
    got = np.array([[r[l] for l in c["labels"]] for r in res], dtype=np.float32)
    assert got.shape == c["scores"].shape
    assert list(res[0].keys()) == c["labels"]
    np.testing.assert_allclose(got, c["scores"], rtol=0, atol=1e-6)


def test_stream_mixed_lengths_matches_reference_plumbing():
    c = load_case("stream_mixed")
    hs = {n: head(n) for n in c["names"]}
    om = streaming.OracleModel(emb_weights(), hs, class_mapping(c["names"]), feature_init=c["feature_init"])
    pos, rows = 0, []
    for n in c["lens"]:
        r = om.predict(c["pcm"][pos:pos + n])
        pos += n
        rows.append([r[l] for l in c["labels"]])
    np.testing.assert_allclose(np.array(rows, np.float32), c["scores"], atol=1e-6)
    np.testing.assert_allclose(om.preprocessor.melspectrogram_buffer[-76:], c["mel_tail"], atol=1e-5)
    np.testing.assert_allclose(om.preprocessor.feature_buffer[-34:], c["feat_tail"], atol=1e-5)


def test_embed_clips_golden():
    c = load_case("embed_clips")
    got = np.stack([streaming.embeddings_of_clip(emb_weights(), p) for p in c["pcm"]])
    np.testing.assert_allclose(got, c["embeddings"], atol=1e-5)


def test_mel_against_torch_stft_and_torchaudio():
    torchaudio = pytest.importorskip("torchaudio")
    rng = np.random.default_rng(3)
    for amp in (300, 20000):
        x = np.clip(rng.normal(0, amp, 8000), -32768, 32767).astype(np.int16)
        st = torch.stft(torch.tensor(x.astype(np.float64)), 512, hop_length=160, win_length=512,
                        window=torch.tensor(mel.hann_window_padded()), center=False, return_complex=True)
        fb = torchaudio.functional.melscale_fbanks(257, 60.0, 3800.0, 32, 16000, norm="slaney", mel_scale="slaney").double()
        db = 10 * torch.log10(torch.clamp((st.abs() ** 2).T @ fb, min=1e-10))
        db = torch.maximum(db, db.max() - 80)
        np.testing.assert_allclose(mel.melspectrogram_raw(x, np.float64), db.numpy(), atol=1e-3)
        np.testing.assert_allclose(mel.melspectrogram_raw(x), db.numpy(), atol=2e-3)
    assert np.abs(mel.mel_filterbank() - fb.numpy()).max() < 1e-7


def test_mel_frame_counts_and_silence_floor():
    assert [mel.n_frames(n) for n in (1760, 1280, 3040, 32000, 64000)] == [8, 5, 16, 197, 397]
    m = mel.melspectrogram(np.zeros(1760, np.int16))
    assert m.shape == (8, 32) and np.allclose(m, -8.0)          # SURVEY.md App. A.8
    with pytest.raises(ValueError):
        mel.melspectrogram_raw(np.zeros(100, np.int16))


def test_cnn_against_torch_conv2d_and_mac_count():
    w = emb_weights()
    rng = np.random.default_rng(1)
    wins = rng.normal(8, 2, (3, 76, 32)).astype(np.float32)
    x = torch.tensor(wins)[:, None].double()
    macs = 0
    for li, (kh, kw, cin, cout, pool) in enumerate(embedding.LAYERS):
        k = torch.tensor(w["conv"][li]).double().permute(3, 2, 0, 1)
        x = torch.nn.functional.conv2d(x, k, padding=(0, 1 if kw == 3 else 0))
        macs += x.shape[2] * x.shape[3] * kh * kw * cin * cout
        if li == 0:
            x = x.relu()
        if li < 19:
            g, b, m, v = [torch.tensor(a).double()[None, :, None, None] for a in w["bn"][li]]
            x = (x - m) / torch.sqrt(v + 1e-3) * g + b
            x = torch.clamp(torch.maximum(float(embedding.LEAK) * x, x), min=float(embedding.FLOOR))
        if pool:
            x = torch.nn.functional.max_pool2d(x, pool, pool)
    assert macs == embedding.MACS_PER_WINDOW == 41955840          # SURVEY.md App. B total
    assert x.shape == (3, 96, 1, 1)
    np.testing.assert_allclose(embedding.embed_windows(w, wins), x[:, :, 0, 0].numpy(), atol=2e-5)


def test_cnn_fully_convolutional_identity():
    """SURVEY.md F10: one pass over [T,32] == the overlapping 76-row windows."""
    w = emb_weights()
    m = mel.melspectrogram(np.random.default_rng(2).integers(-1000, 1000, 32000).astype(np.int16))
    full = embedding.forward(w, m[None])[0]
    wins = np.stack([m[i:i + 76] for i in range(0, m.shape[0] - 75, 8)])
    assert full.shape == (16, 96)
    np.testing.assert_allclose(full, embedding.embed_windows(w, wins), atol=1e-6)


def test_heads_shapes_and_ranges():
    rng = np.random.default_rng(0)
    f16 = rng.normal(0, 1, (5, 16, 96)).astype(np.float32)
    f34 = rng.normal(0, 1, (5, 34, 96)).astype(np.float32)
    a = heads.forward(head("alexa_v0.1"), f16)
    t = heads.forward(head("timer_v0.1"), f34)
    assert a.shape == (5, 1) and np.all((a > 0) & (a < 1))
    assert t.shape == (5, 7) and np.allclose(t.sum(axis=1), 1.0, atol=1e-6)
    # torch reference of the LayerNorm head
    h = head("big_v0.1")
    x = torch.tensor(f16.reshape(5, -1)).double()
    for i, lay in enumerate(h["layers"]):
        x = x @ torch.tensor(lay["W"]).double() + torch.tensor(lay["b"]).double()
        if i < len(h["layers"]) - 1:
            x = torch.nn.functional.layer_norm(x, (x.shape[1],), torch.tensor(lay["ln"][0]).double(),
                                               torch.tensor(lay["ln"][1]).double(), 1e-5).relu()
    np.testing.assert_allclose(heads.forward(h, f16), torch.sigmoid(x).numpy(), atol=1e-6)


def test_stream_features_matches_state_machine_call_by_call():
    """streaming.stream_features (one CNN pass over a segment's mel history) against OracleAudioFeatures fed call by
    call: 46 calls of 1, 2 and 3 chunks, a reset to 120 init rows after call 27, quiet / loud / silent / gated audio.
    The embeddings each call appends and the 120-row feature_buffer must agree; the two differ only in NumPy's
    summation order (measured worst 4.3e-6; gate ~5x)."""
    rng = np.random.default_rng(4)
    plan = [int(x) for x in rng.choice([1, 2, 3], 46)]
    plan[:3] = [3, 1, 2]
    plan[27:29] = [2, 1]                                     # a multi-chunk first call after the reset
    n = sum(plan) * 1280
    pcm = rng.normal(0, 3000, n) * np.repeat(rng.choice([0.0, 0.1, 1.0, 8.0], n // 4000 + 1), 4000)[:n]
    pcm = np.clip(pcm, -32768, 32767).astype(np.int16)
    fi = rng.normal(0, 1, (41, 96)).astype(np.float32)
    fi2 = rng.normal(0, 1, (120, 96)).astype(np.float32)
    rows, ends, starts = streaming.stream_features(emb_weights(), pcm, plan, fi, resets={27: fi2})
    assert rows.shape == (41 + 120 + sum(plan), 96)
    o = streaming.OracleAudioFeatures(emb_weights(), feature_init=fi)
    pos, worst_emb, worst_buf = 0, 0.0, 0.0
    for k, nch in enumerate(plan):
        if k == 27:
            o.reset(feature_init=fi2)
        assert o(pcm[pos:pos + nch * 1280]) == nch * 1280
        pos += nch * 1280
        assert starts[k] == (0 if k < 27 else 41 + sum(plan[:27]))
        assert ends[k] - starts[k] == (41 + sum(plan[:k + 1]) if k < 27 else 120 + sum(plan[27:k + 1]))
        new = rows[ends[k] - nch:ends[k]]
        worst_emb = max(worst_emb, float(np.abs(new - o.feature_buffer[-nch:]).max()))
        buf = rows[max(starts[k], ends[k] - 120):ends[k]]
        assert buf.shape == o.feature_buffer.shape
        worst_buf = max(worst_buf, float(np.abs(buf - o.feature_buffer).max()))
    print(f"stream_features vs OracleAudioFeatures: embeddings {worst_emb:.2e}, feature_buffer {worst_buf:.2e}")
    assert worst_emb < 2e-5 and worst_buf < 2e-5
    assert np.array_equal(rows[:41], fi) and np.array_equal(rows[starts[27]:starts[27] + 120], fi2)


def test_first_chunk_yields_five_frames_and_ones_ring():
    """SURVEY.md F8 / Appendix D.1."""
    af = streaming.OracleAudioFeatures(emb_weights())
    assert af.melspectrogram_buffer.shape == (76, 32) and np.all(af.melspectrogram_buffer == 1.0)
    assert af.feature_buffer.shape == (41, 96)
    rng = np.random.default_rng(0)
    assert af(rng.integers(-1000, 1000, 1280).astype(np.int16)) == 1280
    assert af.melspectrogram_buffer.shape[0] == 81 and af.feature_buffer.shape[0] == 42
    assert af(rng.integers(-1000, 1000, 1280).astype(np.int16)) == 1280
    assert af.melspectrogram_buffer.shape[0] == 89
    assert af(rng.integers(-1000, 1000, 500).astype(np.int16)) == 500
