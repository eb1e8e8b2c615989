"""not-gpu tests: the C-ABI library loads and exports every symbol of include/owwb200.h; weight
packing; registry; and the host-side Model logic driven through a fake (oracle-backed) context
against the golden vectors made from the reference plumbing."""
import ctypes
import os
import re

import numpy as np
import pytest

import openwakeword_b200 as owb
from openwakeword_b200 import _native, weights as W, registry
from openwakeword_b200.utils import re_arg
from helpers import emb_weights, head, class_mapping, golden_cases, load_case, TIMER_MAP
import fake_backend

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol(built_library):
    hdr = open(os.path.join(ROOT, "include", "owwb200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(oww_[a-z_0-9]+)\s*\(", hdr))
    assert declared, "no prototypes found"
    assert declared == set(_native.EXPORTED_SYMBOLS)
    raw = ctypes.CDLL(_native.LIB_PATH)
    for name in declared:
        assert hasattr(raw, name), name
    assert b"sm_100a" in built_library.oww_version()


def test_create_fails_loudly_without_gpu(built_library):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(_native.NativeError):
        _native.Context()
    with pytest.raises(_native.NativeError):      # no silent CPU fallback behind the public API either
        owb.Model(wakeword_models=[{"name": "a", "head": head("alexa_v0.1")}], embedding_model_path="synthetic:0")


def test_embedding_blob_layout_and_param_count():
    w = emb_weights()
    n_conv = sum(a.size for a in w["conv"])
    n_bn = sum(4 * p[0].size for p in w["bn"])
    assert n_conv == 326808 and n_conv + n_bn == W.N_EMBEDDING_PARAMS        # nb/conv:859
    blob = W.pack_embedding_blob(w)
    assert blob.dtype == np.float32 and blob.size == n_conv + 2 * sum(l[3] for l in W.EMBEDDING_LAYERS)
    back = fake_backend.unpack_embedding_blob(blob)
    from oracle import embedding
    x = np.random.default_rng(0).normal(8, 2, (2, 76, 32)).astype(np.float32)
    np.testing.assert_allclose(embedding.embed_windows(back, x), embedding.embed_windows(w, x), atol=1e-4)


def test_head_blob_roundtrip(tmp_path):
    for name in ("alexa_v0.1", "timer_v0.1", "big_v0.1"):
        h = head(name)
        n_in, dims, ln, fin = W.head_desc(h)
        assert dims[0] == n_in * 96
        back = fake_backend.unpack_head_blob(n_in, dims, ln, fin, W.pack_head_blob(h))
        from oracle import heads
        f = np.random.default_rng(1).normal(0, 1, (3, n_in, 96)).astype(np.float32)
        np.testing.assert_array_equal(heads.forward(back, f), heads.forward(h, f))
        p = str(tmp_path / (name + ".npz"))
        W.save_head(p, h, TIMER_MAP if name.startswith("timer") else None)
        h2, cm = W.load_head(p)
        np.testing.assert_array_equal(heads.forward(h2, f), heads.forward(h, f))
        assert (cm == TIMER_MAP) if name.startswith("timer") else cm is None


def test_registry_matches_reference_names():
    assert list(registry.MODELS) == ["alexa", "hey_mycroft", "hey_jarvis", "hey_rhasspy", "timer", "weather"]
    assert registry.model_class_mappings["timer"]["6"] == "1_hour_timer"
    assert len(owb.get_pretrained_model_paths()) == 6


def test_re_arg():
    @re_arg({"old": "new"})
    def f(new=1):
        return new
    assert f(old=5) == 5 and f(new=6) == 6


@pytest.fixture
def fake_ctx(monkeypatch):
    monkeypatch.setattr(_native, "Context", fake_backend.FakeContext)
    yield


def _model(c, **kw):
    specs = [{"name": n, "head": head(n), "class_mapping": class_mapping([n]).get(n)} for n in c["names"]]
    return owb.Model(wakeword_models=specs, embedding_model_path=emb_weights(int(c["emb_seed"])),
                     feature_init=c["feature_init"], max_chunks=8, **kw)


@pytest.mark.parametrize("tag", golden_cases("predict_clip"))
def test_model_host_logic_on_golden(fake_ctx, tag):
    c = load_case(tag)
    m = _model(c)
    res = m.predict_clip(c["pcm"], padding=int(c["padding"]), chunk_size=int(c["chunk"]), **c["kw"])
    assert list(res[0].keys()) == c["labels"]
    got = np.array([[r[l] for l in c["labels"]] for r in res], dtype=np.float32)
    np.testing.assert_allclose(got, c["scores"], atol=1e-5)


def test_model_stream_mixed(fake_ctx):
    c = load_case("stream_mixed")
    c["emb_seed"] = 0
    m = _model(c)
    pos, rows = 0, []
    for n in c["lens"]:
        r = m.predict(c["pcm"][pos:pos + n])
        pos += n
        rows.append([r[l] for l in c["labels"]])
    np.testing.assert_allclose(np.array(rows, np.float32), c["scores"], atol=1e-5)
    np.testing.assert_allclose(m.preprocessor.melspectrogram_buffer, c["mel_tail"], atol=1e-4)
    np.testing.assert_allclose(m.preprocessor.get_features(34)[0], c["feat_tail"], atol=1e-4)
    assert len(m.prediction_buffer[c["labels"][0]]) == len(c["lens"])


def test_model_errors_match_reference(fake_ctx):
    c = load_case("alexa_c1280")
    m = _model(c)
    with pytest.raises(ValueError):
        m.predict([0] * 1280)                                  # model.py:262-263
    with pytest.raises(ValueError):
        m.predict(np.zeros(1280), patience={"alexa_v0.1": 3})   # model.py:341-343
    with pytest.raises(ValueError):
        m.predict(np.zeros(1280, np.int16), patience={"alexa_v0.1": 3}, threshold={"alexa_v0.1": 0.5}, debounce_time=1.0)
    with pytest.raises(ValueError):
        owb.Model(wakeword_models=["no such model"], embedding_model_path="synthetic:0")   # model.py:96-97
    with pytest.raises(ValueError):
        owb.Model(wakeword_models=[{"name": "a", "head": head("alexa_v0.1")}], inference_framework="onnx")
    with pytest.raises(ValueError):
        m.preprocessor._get_melspectrogram(np.zeros(1280, np.float32))     # utils.py:195-197
    r = m.predict(np.zeros(1280))                              # float64 zeros accepted (tests/test_models.py:302-316)
    assert set(r) == {"alexa_v0.1"}
    r, t = m.predict(np.zeros(1280, np.int16), timing=True)
    assert "preprocessor" in t["models"] and "alexa_v0.1" in t["models"]
    assert m.get_parent_model_from_label("alexa_v0.1") == "alexa_v0.1"


def test_model_rejects_heads_wider_than_the_feature_buffer(fake_ctx):
    """oww_add_head bounds n_in by the reference's 120-row feature buffer (a wider window would read ring slots that
    hold newer rows); the fake context keeps the same contract, so Model sees the same error on both."""
    hdr = open(os.path.join(ROOT, "include", "owwb200.h")).read()
    assert re.search(r"#define\s+OWW_MAX_HEAD_FRAMES\s+(\d+)", hdr).group(1) == str(fake_backend.MAX_HEAD_FRAMES) == "120"
    wide = W.synthetic_head(n_in=121, hidden=8, seed=2)
    with pytest.raises(_native.NativeError, match="n_in=121 exceeds the reference's 120-row feature buffer"):
        owb.Model(wakeword_models=[{"name": "wide", "head": wide}], embedding_model_path=emb_weights())
    fi = np.random.default_rng(0).normal(0, 1, (120, 96)).astype(np.float32)
    m = owb.Model(wakeword_models=[{"name": "w120", "head": W.synthetic_head(n_in=120, hidden=8, seed=2)}],
                  embedding_model_path=emb_weights(), feature_init=fi)
    assert m.model_inputs["w120"] == 120
    assert set(m.predict(np.zeros(1280, np.int16))) == {"w120"}


def test_multi_stream_batch_equals_singles(fake_ctx):
    rng = np.random.default_rng(0)
    names = ["alexa_v0.1", "timer_v0.1"]
    specs = [{"name": n, "head": head(n), "class_mapping": class_mapping([n]).get(n)} for n in names]
    fi = rng.normal(0, 1, (41, 96)).astype(np.float32)
    pcm = rng.integers(-3000, 3000, (3, 1280 * 7)).astype(np.int16)
    mb = owb.Model(wakeword_models=specs, embedding_model_path=emb_weights(), feature_init=fi, n_streams=3)
    singles = [owb.Model(wakeword_models=specs, embedding_model_path=emb_weights(), feature_init=fi) for _ in range(3)]
    for s in range(7):
        rb = mb.predict(pcm[:, s * 1280:(s + 1) * 1280])
        for b in range(3):
            r1 = singles[b].predict(pcm[b, s * 1280:(s + 1) * 1280])
            for k in r1:
                assert abs(r1[k] - rb[k][b]) < 1e-6
    assert "1_hour_timer" in rb and rb["alexa_v0.1"].shape == (3,)


def test_model_loads_reference_style_onnx_files(fake_ctx, tmp_path):
    """wakeword_models given as .onnx paths (key = basename, model.py:91-92) + embedding_model.onnx, no onnx package."""
    from openwakeword_b200 import onnx_io
    c = load_case("alexa_c1280")
    hp = str(tmp_path / "alexa_v0.1.onnx")
    ep = str(tmp_path / "embedding_model.onnx")
    onnx_io.write_head_onnx(hp, head("alexa_v0.1"))
    onnx_io.write_embedding_onnx(ep, emb_weights())
    m = owb.Model(wakeword_models=[hp], embedding_model_path=ep, melspec_model_path=str(tmp_path / "melspectrogram.onnx"),
                  feature_init=c["feature_init"])
    assert list(m.models) == ["alexa_v0.1"] and m.model_inputs["alexa_v0.1"] == 16 and m.model_outputs["alexa_v0.1"] == 1
    res = m.predict_clip(c["pcm"])
    got = np.array([[r[l] for l in c["labels"]] for r in res], dtype=np.float32)
    np.testing.assert_allclose(got, c["scores"], atol=1e-5)
    with pytest.raises(ValueError):
        owb.Model(wakeword_models=[str(tmp_path / "x.tflite")], embedding_model_path=ep)


def _oracle_embed_clips(self, x, batch_size=128, ncpu=1):
    """AudioFeatures.embed_clips restated on the oracle (the device call needs a GPU)."""
    from oracle import embedding as oe, mel as om
    x = np.asarray(x)
    if x.dtype != np.int16:
        raise ValueError("Input data must be 16-bit integers.")
    w = emb_weights()
    out = []
    for clip in x:
        m = om.melspectrogram(clip)
        wins = np.stack([m[8 * i:8 * i + 76] for i in range((m.shape[0] - 76) // 8 + 1)])
        out.append(oe.embed_windows(w, wins))
    return np.stack(out).astype(np.float32)


def test_compute_features_from_generator(fake_ctx, monkeypatch, tmp_path):
    """utils.py:542-601: rows land in generator order, the file is cut to what was produced, an n_total below the
    batch size raises, surplus batches are ignored."""
    monkeypatch.setattr(owb.AudioFeatures, "embed_clips", _oracle_embed_clips)
    rng = np.random.default_rng(2)
    S = 16000
    batches = [rng.integers(-1000, 1000, (3, S)).astype(np.int16) for _ in range(3)]
    F = owb.AudioFeatures(embedding_model_path=emb_weights())
    n_w = F.get_embedding_shape(1.0)[0]
    ref = _oracle_embed_clips(None, np.concatenate(batches))

    f1 = str(tmp_path / "over.npy")                       # n_total over-estimates: 9 of 20 rows produced
    owb.compute_features_from_generator(iter(batches), 20, S, f1, audio_features=F)
    a = np.load(f1)
    assert a.shape == (9, n_w, 96) and a.dtype == np.float32
    np.testing.assert_array_equal(a, ref)

    f2 = str(tmp_path / "under.npy")                      # n_total cuts inside the third batch
    owb.compute_features_from_generator(iter(batches), 7, S, f2, audio_features=F)
    np.testing.assert_array_equal(np.load(f2), ref[:7])

    f3 = str(tmp_path / "bad.npy")
    with pytest.raises(ValueError):
        owb.compute_features_from_generator(iter(batches), 2, S, f3, audio_features=F)
    assert not os.path.exists(f3)


def test_threaded_wav_ingest_keeps_order(tmp_path):
    import wave
    from openwakeword_b200.utils import _read_wavs
    rng = np.random.default_rng(4)
    paths, clips = [], []
    for i in range(9):
        c = rng.integers(-3000, 3000, 2000 + 37 * i).astype(np.int16)
        p = str(tmp_path / f"c{i}.wav")
        with wave.open(p, "wb") as f:
            f.setnchannels(1); f.setsampwidth(2); f.setframerate(16000); f.writeframes(c.tobytes())
        paths.append(p); clips.append(c)
    for n in (1, 4):
        got = _read_wavs(paths, n)
        assert all(np.array_equal(g, c) for g, c in zip(got, clips))
    bad = str(tmp_path / "stereo.wav")
    with wave.open(bad, "wb") as f:
        f.setnchannels(2); f.setsampwidth(2); f.setframerate(16000); f.writeframes(np.zeros(64, np.int16).tobytes())
    with pytest.raises(ValueError):
        _read_wavs(paths + [bad], 4)


def test_get_positive_prediction_frames(fake_ctx, tmp_path):
    """model.py:428-478 / tests/test_models.py:323-330: frames at or above the threshold come back as the head's input
    features (or the 4 s audio context); an unreachable threshold gives an empty dict."""
    import wave
    c = load_case("alexa_c1280")
    m = _model(c)
    rng = np.random.default_rng(8)
    pcm = rng.integers(-1000, 1000, 16000 * 5 + 640).astype(np.int16)
    path = str(tmp_path / "clip.wav")
    with wave.open(path, "wb") as f:
        f.setnchannels(1); f.setsampwidth(2); f.setframerate(16000); f.writeframes(pcm.tobytes())
    n_steps = len(range(0, pcm.shape[0] - 1280, 1280))
    name = c["names"][0]
    feats = m._get_positive_prediction_frames(path, threshold=0.0)
    assert list(feats) == [name]
    assert feats[name].shape == (n_steps, m.model_inputs[name], 96)
    m.reset(c["feature_init"])
    audio = m._get_positive_prediction_frames(path, threshold=0.0, return_type="audio")
    n_full = sum(1 for i in range(0, pcm.shape[0] - 1280, 1280) if i - 48000 >= 0 and i + 16000 <= pcm.shape[0])
    assert audio[name].shape == (n_full, 64000)
    first = next(i for i in range(0, pcm.shape[0] - 1280, 1280) if i - 48000 >= 0)
    np.testing.assert_array_equal(audio[name][0], pcm[first - 48000:first + 16000])
    m.reset(c["feature_init"])
    assert m._get_positive_prediction_frames(path, threshold=1.5) == {}
    with pytest.raises(ValueError):
        m._get_positive_prediction_frames(path, return_type="spectrogram")


class _ConstVerifier:
    """Stands in for the scikit-learn pipeline of custom_verifier_model.py: constant P(positive)."""

    def __init__(self, p):
        self.p = p
        self.calls = 0

    def predict_proba(self, feats):
        self.calls += 1
        assert feats.shape[0] == 1 and feats.shape[2] == 96
        return np.array([[1.0 - self.p, self.p]])


def test_custom_verifier_hook(fake_ctx, tmp_path):
    """model.py:175-195,319-328: a verifier pickled per base model replaces that model's score whenever the base score
    reaches custom_verifier_threshold; keys that match no loaded model raise."""
    import pickle
    c = load_case("alexa_c1280")
    name = c["names"][0]
    path = str(tmp_path / "verifier.pkl")
    with open(path, "wb") as f:
        pickle.dump(_ConstVerifier(0.7), f)
    m = _model(c, custom_verifier_models={name: path}, custom_verifier_threshold=0.0)
    rng = np.random.default_rng(1)
    scores = [m.predict(rng.integers(-1000, 1000, 1280).astype(np.int16))[name] for _ in range(8)]
    assert scores[:5] == [0.0] * 5                          # first-five zeroing still applies (model.py:330-333)
    assert all(abs(s - 0.7) < 1e-6 for s in scores[5:])
    plain = _model(c)
    rng = np.random.default_rng(1)
    base = [plain.predict(rng.integers(-1000, 1000, 1280).astype(np.int16))[name] for _ in range(8)]
    assert any(abs(b - 0.7) > 1e-3 for b in base[5:])        # the replacement really changed something
    high = _model(c, custom_verifier_models={name: path}, custom_verifier_threshold=2.0)   # never reached
    rng = np.random.default_rng(1)
    kept = [high.predict(rng.integers(-1000, 1000, 1280).astype(np.int16))[name] for _ in range(8)]
    assert kept == base
    with pytest.raises(ValueError):
        _model(c, custom_verifier_models={"not_loaded": path})


def test_bench_flop_accounting_matches_survey():
    """bench.py's executed-FLOP model: SURVEY.md Appendix B gives 5 612 544 MAC per incremental frame; layers from
    split_from on take three MMA terms per K step (fp16 hi/lo split operands)."""
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    from oracle import embedding as E
    rows, W, macs = 8, 32, []
    for kh, kw, cin, cout, pool in E.LAYERS:
        macs.append(rows * W * kh * kw * cin * cout)
        if pool:
            rows = max(1, rows // pool[0]); W //= pool[1]
    assert macs == b.INC_MACS and sum(macs) == 5612544
    assert b.exec_flops_per_frame(20) == 2 * 5612544 == b.EXEC_FLOPS_PER_FRAME
    assert b.exec_flops_per_frame(0) == b.exec_flops_per_frame(11) == 2 * (5612544 + 2 * sum(macs[11:]))
    assert b.exec_flops_per_frame(15) == 2 * (5612544 + 2 * sum(macs[15:]))
