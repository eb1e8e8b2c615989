"""A CPU stand-in for ``_native.Context`` used ONLY by the not-gpu tests of the host-side logic
(chunk accumulation, label mapping, patience/debounce, bulk grouping).  It implements the C-ABI
semantics with the oracle so that ``openwakeword_b200.Model`` can be driven on a GPU-less box; the
product never sees it."""
import numpy as np

from oracle import mel as omel, embedding as oemb, heads as oheads, streaming as ostream
from openwakeword_b200 import weights as W
from openwakeword_b200._native import NativeError

MAX_HEAD_FRAMES = 120        # OWW_MAX_HEAD_FRAMES: the rows of the reference's feature buffer


def unpack_embedding_blob(blob):
    conv, scale, bias = [], [], []
    off = 0
    for (kh, kw, cin, cout, _, _) in W.EMBEDDING_LAYERS:
        n = kh * kw * cin * cout
        conv.append(blob[off:off + n].reshape(kh, kw, cin, cout)); off += n
        scale.append(blob[off:off + cout]); off += cout
        bias.append(blob[off:off + cout]); off += cout
    assert off == blob.size
    # express folded scale/bias as a BatchNorm with var = 1-eps, mean = 0
    bn = [(s * np.sqrt(np.float64(1.0)), b, np.zeros_like(b), np.full_like(b, 1.0 - 1e-3)) for s, b in zip(scale[:-1], bias[:-1])]
    return {"conv": conv, "bn": bn}


def unpack_head_blob(n_in, dims, layernorm, final_act, blob):
    layers, off = [], 0
    for i in range(len(dims) - 1):
        din, dout = dims[i], dims[i + 1]
        Wm = blob[off:off + din * dout].reshape(din, dout); off += din * dout
        b = blob[off:off + dout]; off += dout
        ln = None
        if layernorm and i < len(dims) - 2:
            ln = (blob[off:off + dout], blob[off + dout:off + 2 * dout]); off += 2 * dout
        layers.append({"W": Wm, "b": b, "ln": ln})
    assert off == blob.size
    fin = {v: k for k, v in W.FINAL_CODES.items()}[final_act]
    return {"n_in": n_in, "layers": layers, "final": fin}


class FakeContext:
    instances = []

    def __init__(self, device=0, max_chunks=4, cnn_mode=0, window_batch=0, fuse_step=True, split_from=11, **kw):
        self.max_chunks = max_chunks
        self.heads = []
        self.gates = []
        self._n = 0
        self.launch_count = 0
        FakeContext.instances.append(self)

    def load_mel(self, window512=None, mel_fb=None):
        pass

    def load_embedding(self, blob):
        self.emb = unpack_embedding_blob(np.asarray(blob, np.float32))

    def add_head(self, n_in, dims, layernorm, final_act, blob):
        if n_in > MAX_HEAD_FRAMES:                       # oww_add_head's bound (include/owwb200.h)
            raise NativeError(f"libowwb200 error -4: head n_in={n_in} exceeds the reference's "
                              f"{MAX_HEAD_FRAMES}-row feature buffer")
        self.heads.append(unpack_head_blob(n_in, list(dims), layernorm, final_act, np.asarray(blob, np.float32)))
        return len(self.heads) - 1

    def add_gate(self, main_head, verifier_head, threshold=0.5):
        self.gates.append((main_head, verifier_head, float(threshold)))

    def _col0(self, hid):
        return sum(h["layers"][-1]["W"].shape[1] for h in self.heads[:hid])

    @property
    def n_outputs(self):
        return sum(h["layers"][-1]["W"].shape[1] for h in self.heads)

    @property
    def n_streams(self):
        return self._n

    def set_streams(self, n):
        self._n = n
        self.af = [ostream.OracleAudioFeatures(self.emb) for _ in range(n)]

    def reset(self, stream_ids=None, feature_init=None):
        ids = range(self._n) if stream_ids is None else stream_ids
        for b in ids:
            self.af[b].reset(feature_init=np.zeros((41, 96), np.float32) if feature_init is None else feature_init)

    def step_host(self, pcm, n_chunks, scores_out):
        for b in range(self._n):
            got = self.af[b](pcm[b])
            assert got == n_chunks * 1280
            per_chunk = []
            for h in self.heads:
                n_in = h["n_in"]
                g = [oheads.forward(h, self.af[b].get_features(n_in, -n_in - i))[0] for i in range(n_chunks - 1, -1, -1)]
                per_chunk.append(np.stack(g))            # [n_chunks, n_out]
            raw = np.concatenate(per_chunk, axis=1)      # [n_chunks, n_cols]
            for m, v, thr in self.gates:                 # per chunk, before the max over chunks (as the gated graph would)
                cm, cv = self._col0(m), self._col0(v)
                raw[:, cm] = np.where(raw[:, cm] > np.float32(thr), raw[:, cv], raw[:, cm])
            scores_out[b, :raw.shape[1]] = raw.max(axis=0)

    def get_features(self, stream_id, n, back=0):
        fb = self.af[stream_id].feature_buffer
        end = fb.shape[0] - back
        rows = fb[max(end - n, 0):end]
        if rows.shape[0] < n:
            rows = np.vstack((np.zeros((n - rows.shape[0], 96), np.float32), rows))
        return rows.astype(np.float32)

    def get_counts(self, stream_id):
        # the oracle caps its buffers like the reference; uncapped counts are not needed by the host logic under test
        return self.af[stream_id].melspectrogram_buffer.shape[0], self.af[stream_id].feature_buffer.shape[0]

    def get_mel(self, stream_id, n_rows=76):
        return self.af[stream_id].melspectrogram_buffer[-n_rows:].astype(np.float32)
