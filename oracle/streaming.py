"""Streaming state machine restatement (single stream, NumPy).

Restates /root/reference/openwakeword/utils.py:163-178,387-463 (AudioFeatures
buffers, chunk accumulation, per-chunk mel + embedding) and
/root/reference/openwakeword/model.py:232-426 (predict / predict_clip score
assembly and post-processing); SURVEY.md Appendix D.  Written from that
description, array-based (no deques), so it is an independent check of the
reference plumbing: tests/golden/make_golden.py drives the reference's own
classes through a stub onnxruntime and this file must reproduce its scores.
"""
import numpy as np
from . import mel as _mel, embedding as _emb, heads as _heads

CHUNK = 1280
TAIL = 480            # 160*3 extra samples fed to the mel model (utils.py:397)
WINDOW = 76
MEL_CAP = 970         # utils.py:166
FEAT_CAP = 120        # utils.py:170
RAW_CAP = 160000      # utils.py:164
N_INIT_FEATS = 41     # embeddings of 4 s of noise (utils.py:169)


def embeddings_of_clip(emb_weights, pcm, dtype=np.float32):
    """``AudioFeatures._get_embeddings`` (utils.py:225-236): mel of the whole clip,
    76-row windows every 8 rows, CNN per window."""
    spec = _mel.melspectrogram(pcm, dtype)
    wins = [spec[i:i + WINDOW] for i in range(0, spec.shape[0], 8) if spec[i:i + WINDOW].shape[0] == WINDOW]
    return _emb.embed_windows(emb_weights, np.stack(wins), dtype)


def stream_features(emb_weights, pcm, plan, feature_init, resets=None, dtype=np.float32):
    """Every feature row one stream receives, computed in one CNN pass per segment instead of one per window.

    pcm: the stream's samples (sum(plan) * 1280 of them); plan: chunks per call; feature_init: rows the stream starts
    with; resets: {call index: init rows} - the stream is reset (``OracleAudioFeatures.reset``) just before that call.
    The mel history of a segment is built as ``OracleAudioFeatures.__call__`` builds it: ones(76, 32), then per call the
    mel of the last n*1280+480 samples (at most the segment's samples: 8n-3 rows on a fresh stream's first call, 8n after),
    each call with its own -80 dB clamp.  The windows of the streaming state machine end at the history's end minus
    multiples of 8, i.e. they start at rows 5, 13, 21, ...; the CNN's pooling strides total 8, so one
    ``embedding.forward`` over history[5:] yields all of them.

    Returns (rows, ends, starts): rows [N, 96] float32 in the order the stream's feature ring receives them, every
    segment's init rows included; after call k the stream's buffer is rows[starts[k]:ends[k]] (before the reference's
    120-row cap), so a head of n_in frames scores chunk i (0 = newest) of call k on rows[ends[k]-i-n_in : ends[k]-i]."""
    resets = dict(resets or {})
    pcm = np.asarray(pcm)
    assert pcm.shape[0] == sum(plan) * CHUNK
    bounds = sorted(set([0] + [k for k in resets if 0 < k < len(plan)])) + [len(plan)]
    rows, ends, starts = [], [], []
    n_rows, pos = 0, 0
    for a, b in zip(bounds[:-1], bounds[1:]):
        init = np.asarray(resets.get(a, feature_init), np.float32).reshape(-1, 96)
        start = n_rows
        rows.append(init)
        n_rows += init.shape[0]
        hist = [np.ones((WINDOW, 32), np.float32)]
        seg0 = pos
        for k in range(a, b):
            pos += plan[k] * CHUNK
            hist.append(_mel.melspectrogram(pcm[max(seg0, pos - plan[k] * CHUNK - TAIL):pos], dtype))
        h = np.concatenate(hist)[5:]
        emb = _emb.forward(emb_weights, h[None], dtype)[0]
        assert emb.shape[0] == sum(plan[a:b])
        rows.append(emb)
        for k in range(a, b):
            n_rows += plan[k]
            ends.append(n_rows)
            starts.append(start)
    return np.concatenate(rows).astype(np.float32), np.array(ends), np.array(starts)


class OracleAudioFeatures:
    def __init__(self, emb_weights, feature_init=None, init_noise=None, dtype=np.float32):
        self.w = emb_weights
        self.dtype = dtype
        self._feature_init = feature_init
        self._init_noise = init_noise
        self.reset()

    def reset(self, feature_init=None, init_noise=None):
        self.raw = np.zeros(0, dtype=np.int16)
        self.melspectrogram_buffer = np.ones((WINDOW, 32), dtype=np.float32)
        self.accumulated_samples = 0
        self.remainder = np.zeros(0, dtype=np.int16)
        fi = feature_init if feature_init is not None else self._feature_init
        noise = init_noise if init_noise is not None else self._init_noise
        if fi is not None:
            self.feature_buffer = np.array(fi, dtype=np.float32)
        elif noise is not None:
            self.feature_buffer = embeddings_of_clip(self.w, np.asarray(noise, dtype=np.int16), self.dtype)
        else:
            self.feature_buffer = np.zeros((N_INIT_FEATS, 96), dtype=np.float32)

    def _push_raw(self, x):
        self.raw = np.concatenate((self.raw, x.astype(np.int16)))[-RAW_CAP:]

    def __call__(self, x):
        x = np.asarray(x)
        if self.remainder.shape[0]:
            x = np.concatenate((self.remainder, x))
            self.remainder = np.zeros(0, dtype=np.int16)
        total = self.accumulated_samples + x.shape[0]
        if total >= CHUNK:
            rem = total % CHUNK
            keep = x[:x.shape[0] - rem] if rem else x
            self._push_raw(keep)
            self.accumulated_samples += keep.shape[0]
            self.remainder = x[x.shape[0] - rem:] if rem else np.zeros(0, dtype=np.int16)
        else:
            self.accumulated_samples += x.shape[0]
            self._push_raw(x)
        processed = 0
        acc = self.accumulated_samples
        if acc >= CHUNK and acc % CHUNK == 0:
            if self.raw.shape[0] < 400:
                raise ValueError("need >= 400 buffered samples")
            seg = self.raw[-(acc + TAIL):]
            self.melspectrogram_buffer = np.vstack(
                (self.melspectrogram_buffer, _mel.melspectrogram(seg, self.dtype)))[-MEL_CAP:]
            nchunk = acc // CHUNK
            for i in range(nchunk - 1, -1, -1):
                end = self.melspectrogram_buffer.shape[0] - 8 * i
                win = self.melspectrogram_buffer[max(end - WINDOW, 0):end]
                if win.shape[0] == WINDOW:
                    e = _emb.embed_windows(self.w, win[None].astype(np.float32), self.dtype)
                    self.feature_buffer = np.vstack((self.feature_buffer, e))
            processed = acc
            self.accumulated_samples = 0
        self.feature_buffer = self.feature_buffer[-FEAT_CAP:]
        return processed if processed else self.accumulated_samples

    def get_features(self, n, start_ndx=-1):
        fb = self.feature_buffer
        if start_ndx != -1:
            end = start_ndx + int(n) if start_ndx + n != 0 else fb.shape[0]
            return fb[start_ndx:end][None].astype(np.float32)
        return fb[-int(n):][None].astype(np.float32)


def _n_out(h):
    net = h["main"] if "verifier" in h else h      # gated pair (hey_jarvis structure): one output, the gated score
    return net["layers"][-1]["W"].shape[1]


class OracleModel:
    """heads: ordered {name: head dict}; class_mapping: {name: {"1": label}} for
    multi-class heads (model.py:177-182)."""

    def __init__(self, emb_weights, heads, class_mapping=None, feature_init=None,
                 init_noise=None, dtype=np.float32):
        self.heads = heads
        self.dtype = dtype
        self.class_mapping = {}
        for name, h in heads.items():
            n_out = _n_out(h)
            if class_mapping and name in class_mapping:
                self.class_mapping[name] = class_mapping[name]
            else:
                self.class_mapping[name] = {str(i): str(i) for i in range(n_out)}
        self.preprocessor = OracleAudioFeatures(emb_weights, feature_init, init_noise, dtype)
        self.prediction_buffer = {}

    def reset(self, feature_init=None, init_noise=None):
        self.prediction_buffer = {}
        self.preprocessor.reset(feature_init, init_noise)

    def _buf(self, k):
        return self.prediction_buffer.setdefault(k, [])

    def _parent(self, label):
        parent = ""
        for m in self.class_mapping:
            if label in self.class_mapping[m].values():
                parent = m
            elif label == m:
                parent = m
        return parent

    def predict(self, x, patience=None, threshold=None, debounce_time=0.0):
        patience = patience or {}
        threshold = threshold or {}
        n = self.preprocessor(x)
        out = {}
        for name, h in self.heads.items():
            n_in = h["n_in"]
            n_out = _n_out(h)
            if n > CHUNK:
                g = [_heads.forward(h, self.preprocessor.get_features(n_in, -n_in - i), self.dtype)[0]
                     for i in range(n // CHUNK - 1, -1, -1)]
                p = np.max(np.stack(g), axis=0)
            elif n == CHUNK:
                p = _heads.forward(h, self.preprocessor.get_features(n_in), self.dtype)[0]
            else:
                if n_out == 1:
                    b = self._buf(name)
                    p = np.array([b[-1] if b else 0.0])
                else:
                    p = np.zeros(max(int(k) for k in self.class_mapping[name]) + 1)
            if n_out == 1:
                out[name] = p[0]
            else:
                for k, lab in self.class_mapping[name].items():
                    out[lab] = p[int(k)]
            for lab in out:                       # model.py:330-333 (all labels so far)
                if len(self._buf(lab)) < 5:
                    out[lab] = 0.0
        if patience or debounce_time > 0:
            if not threshold:
                raise ValueError("threshold required with patience/debounce_time")
            if patience and debounce_time > 0:
                raise ValueError("patience and debounce_time are exclusive")
            for lab in out:
                par = self._parent(lab)
                if out[lab] != 0.0:
                    hist = np.array(self._buf(lab)[-30:])
                    if par in patience:
                        sc = hist[-patience[par]:]
                        if (sc >= threshold[par]).sum() < patience[par]:
                            out[lab] = 0.0
                    elif debounce_time > 0 and par in threshold:
                        nfr = int(np.ceil(debounce_time / (n / 16000)))
                        rec = hist[-nfr:]
                        if out[lab] >= threshold[par] and (rec >= threshold[par]).sum() > 0:
                            out[lab] = 0.0
        for lab in out:
            b = self._buf(lab)
            b.append(out[lab])
            del b[:-30]
        return out

    def predict_clip(self, clip, padding=1, chunk_size=CHUNK, **kw):
        data = np.asarray(clip)
        if padding:
            z = np.zeros(16000 * padding, dtype=np.int16)
            data = np.concatenate((z, data, z))
        return [self.predict(data[i:i + chunk_size], **kw)
                for i in range(0, data.shape[0] - chunk_size, chunk_size)]
