"""Generate tests/golden/*.npz by running the UNMODIFIED reference plumbing.

Needs a checkout of the original openWakeWord project (its ``openwakeword`` package and ``tests/data/*.wav``):
    python tests/golden/make_golden.py <openWakeWord checkout> [--only-new]
Its ``openwakeword`` package is imported with ``oracle.ref_stub_ort`` standing in
for onnxruntime (absent here, SURVEY.md F2), so buffers, windowing, chunk
accumulation and score post-processing are the reference's own code while the
three graphs are evaluated by oracle/{mel,embedding,heads}.py on synthetic seeded
weights (regenerated from the recorded seeds, not stored).  The unseeded
``np.random`` state the reference puts in ``feature_buffer`` (SURVEY.md F6) is
captured and stored as ``feature_init``.
"""
import argparse
import os
import sys
import tempfile
import wave

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from openwakeword_b200 import weights as W          # noqa: E402
from oracle import ref_stub_ort                     # noqa: E402

EMB_SEED = 0
HEAD_SPECS = {   # name -> kwargs of weights.synthetic_head
    "alexa_v0.1": dict(n_in=16, hidden=64, n_blocks=1, n_out=1, layernorm=True, final="sigmoid", seed=1),
    "hey_mycroft_v0.1": dict(n_in=16, hidden=64, n_blocks=1, n_out=1, layernorm=True, final="sigmoid", seed=2),
    "timer_v0.1": dict(n_in=34, hidden=128, n_blocks=1, n_out=7, layernorm=False, final="relu_softmax", seed=9),
    "big_v0.1": dict(n_in=16, hidden=128, n_blocks=2, n_out=1, layernorm=True, final="sigmoid", seed=4),
}
GATED_SPECS = {  # conditional verifier pairs (the hey_jarvis structure): weights.synthetic_gated_head kwargs
    "hey_jarvis_v0.1": dict(seed_main=31, seed_verifier=32, threshold=0.5),
}
TIMER_MAP = {"1": "1_minute_timer", "2": "5_minute_timer", "3": "10_minute_timer",
             "4": "20_minute_timer", "5": "30_minute_timer", "6": "1_hour_timer"}


def read_wav(path):
    with wave.open(path, "rb") as f:
        return np.frombuffer(f.readframes(f.getnframes()), dtype=np.int16).copy()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("reference", help="checkout of the original openWakeWord project")
    ap.add_argument("--only-new", action="store_true", help="keep the committed round-1 fixtures byte-identical")
    args = ap.parse_args()
    out_dir = os.path.dirname(os.path.abspath(__file__))
    emb = W.synthetic_embedding(EMB_SEED)
    heads = {k: W.synthetic_head(**v) for k, v in HEAD_SPECS.items()}
    heads.update({k: W.synthetic_gated_head(**v) for k, v in GATED_SPECS.items()})
    only_new = args.only_new
    ref_stub_ort.install(emb, heads)
    sys.path.insert(0, os.path.abspath(args.reference))
    from openwakeword.model import Model            # the reference, unmodified

    tmp = tempfile.mkdtemp()
    paths = {}
    for k in list(heads) + ["melspectrogram", "embedding_model"]:
        paths[k] = os.path.join(tmp, k + ".onnx")
        open(paths[k], "w").close()

    def make_model(names, seed):
        np.random.seed(seed)
        m = Model(wakeword_models=[paths[n] for n in names],
                  class_mapping_dicts=[({"timer_v0.1": TIMER_MAP} if False else {}) for n in names],
                  inference_framework="onnx",
                  melspec_model_path=paths["melspectrogram"],
                  embedding_model_path=paths["embedding_model"])
        if "timer_v0.1" in names:   # registry mapping is keyed "timer"; give the path-keyed model the same labels
            m.class_mapping["timer_v0.1"] = dict(TIMER_MAP)
        return m, m.preprocessor.feature_buffer.astype(np.float32).copy()

    wavs = {n: read_wav(os.path.join(args.reference, "tests", "data", n + ".wav"))
            for n in ("alexa_test", "hey_mycroft_test", "hey_jane")}
    cases = {}

    def run_clip(tag, names, pcm, seed, chunk, padding=1, new=False, **kw):
        if only_new and not new:
            return
        m, fi = make_model(names, seed)
        res = m.predict_clip(pcm, padding=padding, chunk_size=chunk, **kw)
        labels = list(res[0].keys())
        cases[tag] = dict(kind="predict_clip", names=names, pcm=pcm, feature_init=fi, chunk=chunk,
                          padding=padding, labels=labels, kw=kw,
                          scores=np.array([[r[l] for l in labels] for r in res], dtype=np.float32))
        print(tag, cases[tag]["scores"].shape, float(cases[tag]["scores"].max()))

    all4 = ["alexa_v0.1", "hey_mycroft_v0.1", "timer_v0.1", "big_v0.1"]
    run_clip("alexa_c1280", ["alexa_v0.1"], wavs["alexa_test"], 3, 1280)
    run_clip("alexa_c2560", ["alexa_v0.1"], wavs["alexa_test"], 3, 2560)
    run_clip("alexa_c1024", ["alexa_v0.1"], wavs["alexa_test"], 3, 1024)
    run_clip("alexa_c2048", ["alexa_v0.1"], wavs["alexa_test"], 3, 2048)
    run_clip("alexa_c400", ["alexa_v0.1", "timer_v0.1"], wavs["alexa_test"], 4, 400)
    run_clip("mycroft_all4_c1280", all4, wavs["hey_mycroft_test"], 5, 1280)
    run_clip("mycroft_all4_c3840", all4, wavs["hey_mycroft_test"], 5, 3840)
    run_clip("jane_all4_c1280", all4, wavs["hey_jane"], 6, 1280)
    run_clip("jane_nopad_c1280", ["alexa_v0.1", "timer_v0.1"], wavs["hey_jane"], 7, 1280, padding=0)
    run_clip("jane_debounce", ["hey_mycroft_v0.1"], wavs["hey_jane"], 8, 1280,
             debounce_time=0.5, threshold={"hey_mycroft_v0.1": 0.2})
    run_clip("jane_patience", ["hey_mycroft_v0.1"], wavs["hey_jane"], 8, 1280,
             patience={"hey_mycroft_v0.1": 3}, threshold={"hey_mycroft_v0.1": 0.2})

    # round 2: the conditional verifier pair, one chunk and two chunks per call (gate per chunk, then max)
    run_clip("jarvis_gated_c1280", ["hey_jarvis_v0.1", "alexa_v0.1"], wavs["hey_jane"], 9, 1280, new=True)
    run_clip("jarvis_gated_c2560", ["hey_jarvis_v0.1", "timer_v0.1"], wavs["hey_mycroft_test"], 10, 2560, new=True)
    if only_new:
        return write_cases(cases, out_dir)

    # raw streaming with mixed chunk lengths and a mid-stream reset (state carries over, SURVEY F9)
    rng = np.random.default_rng(11)
    m, fi = make_model(["alexa_v0.1", "timer_v0.1"], 12)
    lens = [1280, 1280, 640, 640, 2560, 100, 1180, 1280, 3000, 840, 1280, 1280, 1280]
    pcm = np.concatenate([rng.integers(-1000, 1000, 6000), (rng.uniform(-1, 1, 6000) * 32767).astype(np.int64),
                          np.zeros(2000, np.int64), rng.normal(0, 8000, sum(lens)).astype(np.int64)])
    pcm = np.clip(pcm, -32768, 32767).astype(np.int16)[:sum(lens)]
    pos, rows = 0, []
    for n in lens:
        r = m.predict(pcm[pos:pos + n])
        pos += n
        rows.append([r[l] for l in r])
    cases["stream_mixed"] = dict(kind="stream", names=["alexa_v0.1", "timer_v0.1"], pcm=pcm, feature_init=fi,
                                 lens=np.array(lens), labels=list(r.keys()),
                                 scores=np.array(rows, dtype=np.float32),
                                 mel_tail=m.preprocessor.melspectrogram_buffer[-76:].astype(np.float32),
                                 feat_tail=m.preprocessor.feature_buffer[-34:].astype(np.float32))
    print("stream_mixed", cases["stream_mixed"]["scores"].shape)

    # embed_clips (utils.py:358-385) through the reference's ThreadPool path
    clips = np.stack([np.clip(rng.normal(0, a, 32000), -32768, 32767).astype(np.int16) for a in (200, 2000, 15000)])
    emb_out = m.preprocessor.embed_clips(clips, batch_size=2, ncpu=1)
    cases["embed_clips"] = dict(kind="embed_clips", pcm=clips, embeddings=emb_out.astype(np.float32))
    print("embed_clips", emb_out.shape)

    write_cases(cases, out_dir)


def write_cases(cases, out_dir):
    for tag, c in cases.items():
        d = {}
        for k, v in c.items():
            if k == "kw":
                for kk, vv in v.items():
                    if isinstance(vv, dict):
                        d["kw_" + kk + "_keys"] = np.array(list(vv.keys()))
                        d["kw_" + kk + "_vals"] = np.array(list(vv.values()), dtype=np.float64)
                    else:
                        d["kw_" + kk] = np.float64(vv)
            elif isinstance(v, (list, tuple)) and v and isinstance(v[0], str):
                d[k] = np.array(v)
            elif isinstance(v, str):
                d[k] = np.str_(v)
            else:
                d[k] = np.asarray(v)
        d["emb_seed"] = np.int64(EMB_SEED)
        np.savez_compressed(os.path.join(out_dir, tag + ".npz"), **d)
    print("wrote", len(cases), "golden files to", out_dir)


if __name__ == "__main__":
    main()
