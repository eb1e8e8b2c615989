// C ABI of libowwb200.so (include/owwb200.h): handle lifetime, weight upload, stream state and the
// orchestration of one streaming step  PCM -> K1 mel -> K2 embedding CNN -> ring append -> K3 heads.
#include "oww_internal.h"
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <algorithm>

static thread_local std::string g_create_error;

int oww_fail(oww_ctx* ctx, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf; else g_create_error = buf;
    return code;
}

namespace {

const int kLayerTable[OWW_N_CONV][6] = {   // kh kw cin cout pool_t pool_f  (SURVEY.md Appendix B)
    {3, 3, 1, 24, 0, 0},
    {1, 3, 24, 24, 0, 0}, {3, 1, 24, 24, 2, 2},
    {1, 3, 24, 48, 0, 0}, {3, 1, 48, 48, 0, 0},
    {1, 3, 48, 48, 0, 0}, {3, 1, 48, 48, 1, 2},
    {1, 3, 48, 72, 0, 0}, {3, 1, 72, 72, 0, 0},
    {1, 3, 72, 72, 0, 0}, {3, 1, 72, 72, 2, 2},
    {1, 3, 72, 96, 0, 0}, {3, 1, 96, 96, 0, 0},
    {1, 3, 96, 96, 0, 0}, {3, 1, 96, 96, 1, 2},
    {1, 3, 96, 96, 0, 0}, {3, 1, 96, 96, 0, 0},
    {1, 3, 96, 96, 0, 0}, {3, 1, 96, 96, 2, 2},
    {3, 1, 96, 96, 0, 0},
};

void fill_layer_table(oww_ctx* ctx) {
    for (int li = 0; li < OWW_N_CONV; ++li) {
        ConvLayer& L = ctx->conv[li];
        L.kh = kLayerTable[li][0]; L.kw = kLayerTable[li][1]; L.cin = kLayerTable[li][2]; L.cout = kLayerTable[li][3];
        L.pool_t = kLayerTable[li][4]; L.pool_f = kLayerTable[li][5];
        L.d_w = L.d_scale = L.d_bias = nullptr;
    }
}

int next_pow2(int v) { int p = 1; while (p < v) p <<= 1; return p; }

__global__ void reset_kernel(const int* ids, int n_ids, int n_streams, int16_t* tail, int* seen, int* mel_count,
                             int* feat_count, float* mel_ring, int mel_rows, float* feat_ring, int feat_rows,
                             const float* feat_init, int n_rows, ResetTails rt) {
    const int j = blockIdx.x;
    const int b = ids ? ids[j] : j;
    if (b < 0 || b >= n_streams) return;
    if (rt.tails) {
        // mode 3: the stream's conv tails become those of the all-ones window (its history after a reset), scattered from
        // the compact per-stream template into the group layout [(r*G + g)*Wp + f] of each tails-bearing tensor
        const int grp = b / rt.G, g = b - grp * rt.G;
        uint4* dst = rt.tails + (int64_t)grp * rt.tail_units;
        for (int k = 0; k < rt.n_tab; ++k) {
            const int off1 = rt.tab[k].x, offG = rt.tab[k].y, cg = rt.tab[k].z, Wp = rt.tab[k].w;
            for (int i = threadIdx.x; i < cg * 2 * Wp; i += blockDim.x) {
                const int pl = i / (2 * Wp), u = i - pl * 2 * Wp, r = u / Wp, f = u - r * Wp;
                dst[offG + pl * (2 * rt.G * Wp) + (r * rt.G + g) * Wp + f] = rt.tmpl[off1 + i];
            }
        }
        // incremental late layers: tails rows of the buffers the next step (and, for single-row tensors, the one after) reads
        for (int k = 0; k < rt.n_late; ++k) {
            const ResetLate& T = rt.late[k];
            for (int i = threadIdx.x; i < T.n_planes * 2 * T.Wp; i += blockDim.x) {
                const int pl = i / (2 * T.Wp), u = i - pl * 2 * T.Wp, r = u / T.Wp, f = u - r * T.Wp;
                const uint4 v = T.tmpl[i];
                if (T.lay.S) {                              // block-major layout (cnn_tc.cu, tc_conv_blk_kernel): no pad column
                    if (f >= T.lay.Wq) continue;
                    T.now[late_unit(T.lay, pl, b, r, f)] = v;
                    if (T.next && r == 1) T.next[late_unit(T.lay, pl, b, 0, f)] = v;
                    continue;
                }
                T.now[(int64_t)pl * T.plane + 8 + ((int64_t)b * T.T_buf + r) * T.Wp + f] = v;
                if (T.next && r == 1) T.next[(int64_t)pl * T.plane + 8 + ((int64_t)b * T.T_buf + 0) * T.Wp + f] = v;
            }
        }
    }
    for (int i = threadIdx.x; i < OWW_TAIL; i += blockDim.x) tail[(int64_t)b * OWW_TAIL + i] = 0;
    float* mr = mel_ring + (int64_t)b * mel_rows * 32;
    for (int i = threadIdx.x; i < mel_rows * 32; i += blockDim.x) mr[i] = 1.0f;     // np.ones((76,32)), utils.py:165
    float* fr = feat_ring + (int64_t)b * feat_rows * 96;
    for (int i = threadIdx.x; i < feat_rows * 96; i += blockDim.x)
        fr[i] = (i < n_rows * 96 && feat_init) ? feat_init[i] : 0.f;
    if (threadIdx.x == 0) {
        seen[b] = 0;
        mel_count[b] = OWW_WINDOW_ROWS;
        feat_count[b] = n_rows;
    }
}

__global__ void gather_chunk_kernel(const int16_t* pcm, int n_clips, int n_samples, int pad, int step, int16_t* out) {
    const int64_t total = (int64_t)n_clips * OWW_SAMPLES_PER_CHUNK;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i / OWW_SAMPLES_PER_CHUNK), k = (int)(i % OWW_SAMPLES_PER_CHUNK);
        const int64_t p = (int64_t)step * OWW_SAMPLES_PER_CHUNK + k - pad;
        out[i] = (p >= 0 && p < n_samples) ? pcm[(int64_t)c * n_samples + p] : (int16_t)0;
    }
}

}  // namespace
// Tails of the all-ones window per tails-bearing tensor, in the compact G = 1 layout, computed once per weight set by
// the full-window tcgen05 kernels (cnn_tc.cu) - the state every freshly reset stream starts from (its mel history IS
// ones(76,32), utils.py:165, and a constant history is shift invariant, so no per-stream re-priming pass is needed).
int oww_inc_build_template(oww_ctx* ctx);
namespace {

void free_streams(oww_ctx* c) {
    cudaFree(c->d_tail); cudaFree(c->d_seen); cudaFree(c->d_mel_count); cudaFree(c->d_feat_count);
    cudaFree(c->d_mel_ring); cudaFree(c->d_feat_ring); cudaFree(c->d_act[0]); cudaFree(c->d_act[1]);
    cudaFree(c->d_emb_tmp); cudaFree(c->d_inc_tails[0]); cudaFree(c->d_inc_tails[1]);
    cudaFree(c->d_reset_ids); cudaFree(c->d_reset_init);
    cudaFree(c->d_scores_tmp);
    oww_heads_grp_drop_mirror(c);
    for (auto& X : c->late_x) for (auto& b : X.buf) { cudaFree(b); b = nullptr; }
    cudaFree(c->d_late_tmp[0]); c->d_late_tmp[0] = nullptr;
    cudaFree(c->d_late_template); c->d_late_template = nullptr;
    c->late_active = false;
    c->d_tail = nullptr; c->d_seen = c->d_mel_count = c->d_feat_count = nullptr;
    c->d_mel_ring = c->d_feat_ring = c->d_act[0] = c->d_act[1] = c->d_emb_tmp = nullptr;
    c->d_inc_tails[0] = c->d_inc_tails[1] = nullptr;
    c->d_reset_ids = nullptr; c->d_reset_init = nullptr;
    c->d_scores_tmp = nullptr; c->scores_tmp_floats = 0;
    c->act_floats = c->emb_tmp_floats = 0;
    c->n_streams = 0;
}

int ensure_act(oww_ctx* ctx, size_t floats) {
    if (ctx->cfg.cnn_mode == OWW_CNN_TC_WINDOW || ctx->cfg.cnn_mode == OWW_CNN_TC_INCREMENTAL) {
        // `floats` is n_windows * 74*32*24 (layer-1 output of the fp32 path): size the fp16 planes for the same windows
        int n_win = (int)(floats / ((size_t)74 * 32 * 24));
        if (n_win < 1) n_win = 1;
        if (n_win > ctx->window_batch) n_win = ctx->window_batch;
        const size_t units = oww_tc_act_units(ctx, n_win);
        if (ctx->tc_act_units < units) {
            cudaFree(ctx->d_tc_act[0]); cudaFree(ctx->d_tc_act[1]);
            ctx->d_tc_act[0] = ctx->d_tc_act[1] = nullptr; ctx->tc_act_units = 0;
            for (int i = 0; i < 2; ++i) {
                OWW_CUDA(ctx, cudaMalloc(&ctx->d_tc_act[i], units * 16));
                OWW_CUDA(ctx, cudaMemset(ctx->d_tc_act[i], 0, units * 16));
            }
            ctx->tc_act_units = units;
        }
    }
    if (ctx->act_floats >= floats) return OWW_OK;
    cudaFree(ctx->d_act[0]); cudaFree(ctx->d_act[1]);
    ctx->d_act[0] = ctx->d_act[1] = nullptr; ctx->act_floats = 0;
    OWW_CUDA(ctx, cudaMalloc(&ctx->d_act[0], floats * sizeof(float)));
    OWW_CUDA(ctx, cudaMalloc(&ctx->d_act[1], floats * sizeof(float)));
    ctx->act_floats = floats;
    return OWW_OK;
}

// grow the fp16 plane scratch of the tensor-core window / clip passes to `units` 16-byte units per buffer
int ensure_tc_units(oww_ctx* ctx, size_t units) {
    if (ctx->tc_act_units >= units) return OWW_OK;
    cudaFree(ctx->d_tc_act[0]); cudaFree(ctx->d_tc_act[1]);
    ctx->d_tc_act[0] = ctx->d_tc_act[1] = nullptr; ctx->tc_act_units = 0;
    for (int i = 0; i < 2; ++i) {
        OWW_CUDA(ctx, cudaMalloc(&ctx->d_tc_act[i], units * 16));
        OWW_CUDA(ctx, cudaMemset(ctx->d_tc_act[i], 0, units * 16));
    }
    ctx->tc_act_units = units;
    return OWW_OK;
}

__global__ void fill_init_rows_kernel(float* feats, int64_t clip_stride, int n_clips, const float* init, int n_rows) {
    const int64_t total = (int64_t)n_clips * n_rows * 24;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c4 = (int)(i % 24);
        const int r = (int)((i / 24) % n_rows);
        const int64_t clip = i / ((int64_t)24 * n_rows);
        reinterpret_cast<float4*>(feats + clip * clip_stride + (int64_t)r * 96)[c4] =
            init ? __ldg(reinterpret_cast<const float4*>(init + (int64_t)r * 96) + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

int ensure_emb_tmp(oww_ctx* ctx, size_t floats) {
    if (ctx->emb_tmp_floats >= floats) return OWW_OK;
    cudaFree(ctx->d_emb_tmp); ctx->d_emb_tmp = nullptr; ctx->emb_tmp_floats = 0;
    OWW_CUDA(ctx, cudaMalloc(&ctx->d_emb_tmp, floats * sizeof(float)));
    ctx->emb_tmp_floats = floats;
    return OWW_OK;
}

int step_core(oww_ctx* ctx, const int16_t* d_pcm, int64_t pcm_stride, int n_chunks, float* d_scores, int out_stride,
              cudaStream_t s) {
    const int B = ctx->n_streams;
    if (B <= 0) return oww_fail(ctx, OWW_EINVAL, "oww_set_streams has not been called");
    if (n_chunks < 1 || n_chunks > ctx->cfg.max_chunks)
        return oww_fail(ctx, OWW_EINVAL, "n_chunks=%d outside [1,%d]", n_chunks, ctx->cfg.max_chunks);
    if (!ctx->mel_loaded || !ctx->emb_loaded) return oww_fail(ctx, OWW_EINVAL, "weights not loaded");
    int rc;
    const long slot = ctx->timing ? ctx->ev_steps % ctx->ev_slots : 0;
    cudaEvent_t* ev = ctx->timing ? &ctx->ev[4 * slot] : nullptr;
    const bool inc = ctx->cfg.cnn_mode == OWW_CNN_TC_INCREMENTAL;
    const FeatSrc fs0{ctx->d_feat_ring, (int64_t)ctx->feat_rows * 96, ctx->d_feat_count, ctx->feat_rows - 1, 0};

    if (inc && n_chunks == 1 && oww_fused_frontend_supported(ctx)) {
        // ---- one chunk: frontend + CNN + ring append of every stream in ONE launch (fresh streams included: a reset
        //      leaves the tails of the all-ones window behind, see reset_kernel) ----
        const bool heads_inside = oww_fused_heads_supported(ctx);
        if (ev) OWW_CUDA(ctx, cudaEventRecord(ev[1], s));
        if ((rc = oww_fused_step(ctx, d_pcm, pcm_stride, d_scores, out_stride, heads_inside, s))) return rc;
        if (ctx->late_active) {
            // cut plan: conv layers >= split_from run as their own launches (split operands) and the embedding is appended here
            if ((rc = oww_late_chain(ctx, ctx->d_emb_tmp, s))) return rc;
            if ((rc = oww_feat_append(ctx, ctx->d_emb_tmp, 1, s))) return rc;
        }
        if (ev) OWW_CUDA(ctx, cudaEventRecord(ev[2], s));
        if (heads_inside) oww_feat16_invalidate(ctx);
        else if ((rc = oww_feat16_advance(ctx, 1, s))) return rc;
        if (!heads_inside && (rc = oww_heads_all(ctx, fs0, B, d_scores, out_stride, 0, s))) return rc;
        if (ev) {
            if (heads_inside) ctx->ev_fused[slot] = 1;
            else { OWW_CUDA(ctx, cudaEventRecord(ev[3], s)); ctx->ev_fused[slot] = 2; }
            ctx->ev_steps++;
        }
        return OWW_OK;
    }

    // ---- general path: separate launches (modes 0 / 2, multi-chunk calls, --no-fuse) ----
    if (ev) { OWW_CUDA(ctx, cudaEventRecord(ev[0], s)); ctx->ev_fused[slot] = 0; }
    MelLaunch m{d_pcm, pcm_stride, n_chunks * OWW_SAMPLES_PER_CHUNK, ctx->d_tail, ctx->d_seen, ctx->d_mel_ring,
                (int64_t)ctx->mel_rows * 32, ctx->mel_rows - 1, ctx->d_mel_count, B, 1, n_chunks};
    if ((rc = oww_mel_launch(ctx, m, s))) return rc;
    if (ev) OWW_CUDA(ctx, cudaEventRecord(ev[1], s));
    WindowSrc ws{ctx->d_mel_ring, (int64_t)ctx->mel_rows * 32, ctx->d_mel_count, ctx->mel_rows - 1, B, n_chunks};
    if (inc) {
        // one incremental launch per chunk on the 8 mel rows that chunk added (a fresh stream's first chunk added 5:
        // the three rows before them are ones of its initial ring, which is what the step then reads)
        for (int i = 0; i < n_chunks; ++i)
            if ((rc = oww_cnn_inc_step(ctx, 8 * (n_chunks - 1 - i), ctx->d_emb_tmp + (size_t)i * B * 96, s))) return rc;
    } else {
        if ((rc = oww_cnn_window(ctx, ws, B * n_chunks, ctx->d_emb_tmp, s, false))) return rc;
    }
    if ((rc = oww_feat_append(ctx, ctx->d_emb_tmp, n_chunks, s))) return rc;
    if (ev) OWW_CUDA(ctx, cudaEventRecord(ev[2], s));
    if ((rc = oww_feat16_advance(ctx, n_chunks, s))) return rc;
    for (int i = n_chunks - 1; i >= 0; --i) {
        FeatSrc fs = fs0; fs.back = i;
        if ((rc = oww_heads_all(ctx, fs, B, d_scores, out_stride, i != n_chunks - 1, s))) return rc;
    }
    if (ev) { OWW_CUDA(ctx, cudaEventRecord(ev[3], s)); ctx->ev_steps++; }
    return OWW_OK;
}

// shared by oww_reset (synchronous) and oww_reset_async: enqueue the state reset of the listed streams on `s`
int reset_enqueue(oww_ctx* ctx, const int32_t* h_stream_ids, int n, const float* h_feature_init, int n_rows, cudaStream_t s) {
    if (ctx->n_streams <= 0) return oww_fail(ctx, OWW_EINVAL, "oww_set_streams has not been called");
    if (n_rows < 0 || n_rows > ctx->feat_rows) return oww_fail(ctx, OWW_EINVAL, "n_rows=%d outside [0,%d]", n_rows, ctx->feat_rows);
    if (!h_stream_ids) n = ctx->n_streams;
    if (n <= 0) return OWW_OK;
    if (n > ctx->n_streams) return oww_fail(ctx, OWW_EINVAL, "more stream ids (%d) than streams (%d)", n, ctx->n_streams);
    if (h_stream_ids) {
        for (int i = 0; i < n; ++i)
            if (h_stream_ids[i] < 0 || h_stream_ids[i] >= ctx->n_streams)
                return oww_fail(ctx, OWW_EINVAL, "stream id %d out of range", h_stream_ids[i]);
        // pageable source: staged by the driver before the call returns; stream-ordered on the device
        OWW_CUDA(ctx, cudaMemcpyAsync(ctx->d_reset_ids, h_stream_ids, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, s));
    }
    const bool have_init = h_feature_init && n_rows > 0;
    if (have_init)
        OWW_CUDA(ctx, cudaMemcpyAsync(ctx->d_reset_init, h_feature_init, (size_t)n_rows * 96 * sizeof(float), cudaMemcpyHostToDevice, s));
    ResetTails rt;
    std::memset(&rt, 0, sizeof(rt));
    if (ctx->cfg.cnn_mode == OWW_CNN_TC_INCREMENTAL) {
        if (!ctx->tails_template_valid) { int rc = oww_inc_build_template(ctx); if (rc) return rc; }
        rt.tails = reinterpret_cast<uint4*>(ctx->d_inc_tails[ctx->inc_cur]);      // the buffer the next step reads
        rt.tmpl = reinterpret_cast<const uint4*>(ctx->d_tails_template);
        rt.G = ctx->inc_plan.G; rt.tail_units = ctx->inc_plan.tail_units; rt.n_tab = ctx->n_tail_tab;
        for (int k = 0; k < ctx->n_tail_tab; ++k) rt.tab[k] = ctx->tail_tab[k];
        if (ctx->late_active) {
            const long k = ctx->late_step;                      // index of the next chunk any stream processes
            for (int l = ctx->split_from; l < OWW_N_CONV; ++l) {
                const oww_ctx::LateTensor& X = ctx->late_x[l];
                if (X.tmpl_off < 0) continue;
                ResetLate& T = rt.late[rt.n_late++];
                T.now = reinterpret_cast<uint4*>(X.buf[k % X.n_buf]);
                T.next = X.n_buf == 3 ? reinterpret_cast<uint4*>(X.buf[(k + 1) % 3]) : nullptr;
                T.tmpl = reinterpret_cast<const uint4*>(ctx->d_late_template) + X.tmpl_off;
                T.plane = X.plane; T.T_buf = X.T_buf; T.Wp = X.W + 1; T.n_planes = 2 * X.cg;
                T.lay = X.lay;
            }
        }
    }
    reset_kernel<<<n, 256, 0, s>>>(h_stream_ids ? ctx->d_reset_ids : nullptr, n, ctx->n_streams, ctx->d_tail, ctx->d_seen,
                                   ctx->d_mel_count, ctx->d_feat_count, ctx->d_mel_ring, ctx->mel_rows, ctx->d_feat_ring,
                                   ctx->feat_rows, have_init ? ctx->d_reset_init : nullptr, n_rows, rt);
    OWW_LAUNCH_CHECK(ctx);
    return oww_feat16_resync(ctx, h_stream_ids ? ctx->d_reset_ids : nullptr, n, s);     // fp16 mirror of the rings (heads_grp.cu)
}

}  // namespace

extern "C" {

const char* oww_version(void) { return "owwb200 0.1 (sm_100a)"; }

const char* oww_last_error(const oww_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int oww_create(const oww_config* cfg, oww_ctx** out) {
    if (!cfg || !out) return oww_fail(nullptr, OWW_EINVAL, "null argument");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return oww_fail(nullptr, OWW_ECUDA, "no CUDA device: %s", e == cudaSuccess ? "count is 0" : cudaGetErrorString(e));
    if (cfg->device < 0 || cfg->device >= ndev) return oww_fail(nullptr, OWW_EINVAL, "device %d out of range", cfg->device);
    if (cfg->cnn_mode != OWW_CNN_FP32_WINDOW && cfg->cnn_mode != OWW_CNN_TC_WINDOW && cfg->cnn_mode != OWW_CNN_TC_INCREMENTAL)
        return oww_fail(nullptr, OWW_EUNSUPPORTED, "cnn_mode %d not built in this version", cfg->cnn_mode);
    oww_ctx* ctx = new (std::nothrow) oww_ctx();
    if (!ctx) return oww_fail(nullptr, OWW_ENOMEM, "out of host memory");
    ctx->cfg = *cfg;
    if (ctx->cfg.max_chunks < 1) ctx->cfg.max_chunks = 1;
    ctx->device = cfg->device;
    ctx->fuse_step = (cfg->reserved[0] & 1) == 0;
    ctx->window_batch = cfg->window_batch > 0 ? cfg->window_batch : (cfg->cnn_mode == OWW_CNN_FP32_WINDOW ? 512 : 1024);
    if ((e = cudaSetDevice(ctx->device)) != cudaSuccess) {
        oww_fail(nullptr, OWW_ECUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
        delete ctx; return OWW_ECUDA;
    }
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, ctx->device);
    ctx->sm_count = prop.multiProcessorCount;
    if (prop.major != 10) {
        oww_fail(nullptr, OWW_EUNSUPPORTED, "device is sm_%d%d; this library is built for sm_100a only", prop.major, prop.minor);
        delete ctx; return OWW_EUNSUPPORTED;
    }
    ctx->tc_heads = (cfg->reserved[0] & 2) == 0;
    ctx->split_from = (cfg->reserved[1] >= 2 && cfg->reserved[1] <= OWW_N_CONV) ? cfg->reserved[1] : 11;
    ctx->tc_heads_terms = (cfg->reserved[0] & 4) ? 1 : 3;
    ctx->grp_heads = (cfg->reserved[0] & 8) == 0;
    ctx->late_blocked_ok = (cfg->reserved[0] & 16) == 0;
    ctx->late_pdl = (cfg->reserved[0] & 32) == 0;
    cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking);
    cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking);
    fill_layer_table(ctx);
    *out = ctx;
    return OWW_OK;
}

void oww_destroy(oww_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->clip_ctx) { oww_ctx* c = ctx->clip_ctx; ctx->clip_ctx = nullptr; free_streams(c);
        cudaStreamDestroy(c->own_stream);
        cudaFree(c->d_tails_template);
        cudaFree(c->d_tc_act[0]); cudaFree(c->d_tc_act[1]);
        cudaFree(c->slot[0].d_pcm); oww_heads_grp_free(c); delete c; }
    free_streams(ctx);
    oww_heads_grp_free(ctx);
    cudaFree(ctx->d_window); cudaFree(ctx->d_twiddle); cudaFree(ctx->d_mel_start); cudaFree(ctx->d_mel_len);
    cudaFree(ctx->d_mel_w); cudaFree(ctx->d_emb_blob); cudaFree(ctx->d_tc_w); cudaFree(ctx->d_tc_sb);
    cudaFree(ctx->d_tc_w3); cudaFree(ctx->d_tc_sb3);
    cudaFree(ctx->d_tc_act[0]); cudaFree(ctx->d_tc_act[1]); cudaFree(ctx->d_inc_w); cudaFree(ctx->d_head_devs);
    for (auto& h : ctx->heads) { cudaFree(h.d_blob); cudaFree(h.d_w1_tc); }
    cudaFree(ctx->d_gates); cudaFree(ctx->d_tails_template); cudaFree(ctx->d_peer_err);
    for (auto& S : ctx->slot) {
        cudaFreeHost(S.h_pcm); cudaFreeHost(S.h_scores); cudaFree(S.d_pcm); cudaFree(S.d_scores);
        if (S.done) cudaEventDestroy(S.done);
        if (S.h2d_done) cudaEventDestroy(S.h2d_done);
    }
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    for (auto e : ctx->ev) cudaEventDestroy(e);
    cudaStreamDestroy(ctx->own_stream);
    delete ctx;
}

int oww_load_embedding(oww_ctx* ctx, const float* h_blob, size_t n_floats) {
    if (!ctx || !h_blob) return oww_fail(ctx, OWW_EINVAL, "null argument");
    size_t need = 0;
    for (int li = 0; li < OWW_N_CONV; ++li) {
        const ConvLayer& L = ctx->conv[li];
        need += (size_t)L.kh * L.kw * L.cin * L.cout + 2 * (size_t)L.cout;
    }
    if (n_floats != need)
        return oww_fail(ctx, OWW_EINVAL, "embedding blob has %zu floats, the reference CNN needs %zu", n_floats, need);
    OWW_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!ctx->d_emb_blob) OWW_CUDA(ctx, cudaMalloc(&ctx->d_emb_blob, need * sizeof(float)));
    OWW_CUDA(ctx, cudaMemcpy(ctx->d_emb_blob, h_blob, need * sizeof(float), cudaMemcpyHostToDevice));
    size_t off = 0;
    for (int li = 0; li < OWW_N_CONV; ++li) {
        ConvLayer& L = ctx->conv[li];
        L.d_w = ctx->d_emb_blob + off; off += (size_t)L.kh * L.kw * L.cin * L.cout;
        L.d_scale = ctx->d_emb_blob + off; off += L.cout;
        L.d_bias = ctx->d_emb_blob + off; off += L.cout;
    }
    ctx->emb_loaded = true;
    ctx->tails_template_valid = false;                 // depends on the weights: rebuilt at the next reset
    int rc = oww_tc_pack_weights(ctx, h_blob);
    if (rc) return rc;
    return oww_inc_setup(ctx, h_blob);
}

int oww_add_head(oww_ctx* ctx, const oww_head_desc* desc, const float* h_blob, size_t n_floats, int* head_id) {
    if (!ctx || !desc || !h_blob) return oww_fail(ctx, OWW_EINVAL, "null argument");
    if (desc->n_layers < 1 || desc->n_layers > OWW_MAX_HEAD_LAYERS)
        return oww_fail(ctx, OWW_EUNSUPPORTED, "head has %d Linear layers (1..%d supported)", desc->n_layers, OWW_MAX_HEAD_LAYERS);
    if (desc->n_in < 1 || desc->dims[0] != desc->n_in * OWW_EMBEDDING_DIM)
        return oww_fail(ctx, OWW_EINVAL, "dims[0]=%d must equal n_in*96=%d", desc->dims[0], desc->n_in * OWW_EMBEDDING_DIM);
    if (desc->n_in > OWW_MAX_HEAD_FRAMES)
        // a chunk `back` rows before the newest reads ring rows count-back-n_in .. count-back-1 (mod feat_rows); with
        // n_in + back > feat_rows the oldest alias newer ones.  feat_rows >= 120 + max_chunks keeps 120-row windows clear.
        return oww_fail(ctx, OWW_EUNSUPPORTED, "head n_in=%d exceeds the reference's %d-row feature buffer",
                        desc->n_in, OWW_MAX_HEAD_FRAMES);
    if (desc->final_act < 0 || desc->final_act > 4) return oww_fail(ctx, OWW_EINVAL, "bad final_act");
    if (ctx->heads.size() >= 16) return oww_fail(ctx, OWW_EUNSUPPORTED, "at most 16 heads per handle");
    Head h;
    h.desc = *desc;
    // Device layout: the caller's tensors in order, each starting on a 16-byte boundary (the fused step kernel streams
    // weight rows with bulk copies, which need 16-byte aligned sources).  `src` walks the packed host blob.
    size_t off = 0, src = 0;
    std::vector<float> staged;
    auto place = [&](size_t n) {
        off = (off + 3) & ~(size_t)3;
        const size_t at = off;
        if (src + n <= n_floats) {
            staged.resize(at + n + 4, 0.f);
            std::memcpy(staged.data() + at, h_blob + src, n * sizeof(float));
        }
        src += n; off += n;
        return at;
    };
    for (int l = 0; l < desc->n_layers; ++l) {
        const int din = desc->dims[l], dout = desc->dims[l + 1];
        if (dout < 1 || dout > 256) return oww_fail(ctx, OWW_EUNSUPPORTED, "layer width %d outside 1..256", dout);
        h.w_off.push_back(place((size_t)din * dout));
        h.b_off.push_back(place(dout));
        if (desc->layernorm && l < desc->n_layers - 1) {
            h.g_off.push_back(place(dout));
            h.h_off.push_back(place(dout));
        } else { h.g_off.push_back(0); h.h_off.push_back(0); }
    }
    if (src != n_floats) return oww_fail(ctx, OWW_EINVAL, "head blob has %zu floats, descriptor needs %zu", n_floats, src);
    OWW_CUDA(ctx, cudaSetDevice(ctx->device));
    OWW_CUDA(ctx, cudaMalloc(&h.d_blob, staged.size() * sizeof(float)));
    OWW_CUDA(ctx, cudaMemcpy(h.d_blob, staged.data(), staged.size() * sizeof(float), cudaMemcpyHostToDevice));
    {   // tensor-core packing of the first layer (heads_tc.cu); heads it does not cover keep tc_ok == false
        int rc = oww_heads_tc_pack(ctx, h, staged.data());
        if (rc) { cudaFree(h.d_blob); return rc; }
    }
    h.n_out = desc->dims[desc->n_layers];
    h.col0 = ctx->n_out_total;
    ctx->n_out_total += h.n_out;
    ctx->max_n_in = std::max(ctx->max_n_in, desc->n_in);
    ctx->heads.push_back(h);
    if (head_id) *head_id = (int)ctx->heads.size() - 1;
    return oww_heads_sync_devs(ctx);
}

int oww_add_gate(oww_ctx* ctx, int main_head, int verifier_head, float threshold) {
    if (!ctx) return OWW_EINVAL;
    const int nh = (int)ctx->heads.size();
    if (main_head < 0 || main_head >= nh || verifier_head < 0 || verifier_head >= nh || main_head == verifier_head)
        return oww_fail(ctx, OWW_EINVAL, "bad head ids %d / %d", main_head, verifier_head);
    if (ctx->heads[main_head].n_out != 1 || ctx->heads[verifier_head].n_out != 1)
        return oww_fail(ctx, OWW_EUNSUPPORTED, "a verifier gate joins two single-output heads");
    if (ctx->gates.size() >= 16) return oww_fail(ctx, OWW_EUNSUPPORTED, "at most 16 gates per handle");
    OWW_CUDA(ctx, cudaSetDevice(ctx->device));
    ctx->gates.push_back(Gate{ctx->heads[main_head].col0, ctx->heads[verifier_head].col0, threshold});
    cudaFree(ctx->d_gates); ctx->d_gates = nullptr;
    OWW_CUDA(ctx, cudaMalloc(&ctx->d_gates, ctx->gates.size() * sizeof(Gate)));
    OWW_CUDA(ctx, cudaMemcpy(ctx->d_gates, ctx->gates.data(), ctx->gates.size() * sizeof(Gate), cudaMemcpyHostToDevice));
    return OWW_OK;
}

int oww_n_heads(const oww_ctx* ctx) { return ctx ? (int)ctx->heads.size() : 0; }
int oww_n_outputs(const oww_ctx* ctx) { return ctx ? ctx->n_out_total : 0; }
int oww_n_streams(const oww_ctx* ctx) { return ctx ? ctx->n_streams : 0; }
uint64_t oww_launch_count(const oww_ctx* ctx) { return ctx ? ctx->launches : 0; }

int oww_melspectrogram(oww_ctx* ctx, const int16_t* d_pcm, int n_clips, int n_samples, float* d_mel, int affine, void* stream) {
    if (!ctx || !d_pcm || !d_mel) return oww_fail(ctx, OWW_EINVAL, "null argument");
    if (n_samples < OWW_FFT_N) return oww_fail(ctx, OWW_EINVAL, "need at least 512 samples, got %d", n_samples);
    OWW_CUDA(ctx, cudaSetDevice(ctx->device));
    const int T = (n_samples - OWW_FFT_N) / OWW_HOP + 1;
    MelLaunch m{d_pcm, (int64_t)n_samples, n_samples, nullptr, nullptr, d_mel, (int64_t)T * 32, -1, nullptr, n_clips,
                affine, 0};
    return oww_mel_launch(ctx, m, (cudaStream_t)stream);
}

int oww_embed_windows(oww_ctx* ctx, const float* d_windows, int n, float* d_emb, void* stream) {
    if (!ctx || !d_windows || !d_emb) return oww_fail(ctx, OWW_EINVAL, "null argument");
    OWW_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = ensure_act(ctx, (size_t)std::min(n, ctx->window_batch) * 74 * 32 * 24);
    if (rc) return rc;
    WindowSrc src{d_windows, (int64_t)OWW_WINDOW_ROWS * 32, nullptr, -1, 0, 0};
    return oww_cnn_window(ctx, src, n, d_emb, (cudaStream_t)stream);
}

int oww_head_predict(oww_ctx* ctx, int head_id, const float* d_feats, int n, float* d_out, void* stream) {
    if (!ctx || !d_feats || !d_out) return oww_fail(ctx, OWW_EINVAL, "null argument");
    if (head_id < 0 || head_id >= (int)ctx->heads.size()) return oww_fail(ctx, OWW_EINVAL, "bad head_id %d", head_id);
    OWW_CUDA(ctx, cudaSetDevice(ctx->device));
    const Head& h = ctx->heads[head_id];
    FeatSrc fs{d_feats, (int64_t)h.desc.n_in * 96, nullptr, -1, 0};
    if (oww_heads_tc_supported(ctx, head_id))
        return oww_heads_tc_launch(ctx, head_id, fs, n, d_out, h.n_out, 0, 0, (cudaStream_t)stream);
    return oww_heads_launch(ctx, head_id, fs, n, d_out, h.n_out, 0, 0, (cudaStream_t)stream);
}

int oww_set_streams(oww_ctx* ctx, int n_streams) {
    if (!ctx || n_streams < 1) return oww_fail(ctx, OWW_EINVAL, "n_streams must be >= 1");
    OWW_CUDA(ctx, cudaSetDevice(ctx->device));
    OWW_CUDA(ctx, cudaDeviceSynchronize());
    free_streams(ctx);
    const int B = n_streams, mc = ctx->cfg.max_chunks;
    ctx->mel_rows = next_pow2(OWW_WINDOW_ROWS + 8 * mc);
    ctx->feat_rows = next_pow2(120 + mc);             // the reference keeps <=120 rows (utils.py:170)
    OWW_CUDA(ctx, cudaMalloc(&ctx->d_tail, (size_t)B * OWW_TAIL * sizeof(int16_t)));
    OWW_CUDA(ctx, cudaMalloc(&ctx->d_seen, (size_t)B * sizeof(int)));
    OWW_CUDA(ctx, cudaMalloc(&ctx->d_mel_count, (size_t)B * sizeof(int)));
    OWW_CUDA(ctx, cudaMalloc(&ctx->d_feat_count, (size_t)B * sizeof(int)));
    OWW_CUDA(ctx, cudaMalloc(&ctx->d_mel_ring, (size_t)B * ctx->mel_rows * 32 * sizeof(float)));
    OWW_CUDA(ctx, cudaMalloc(&ctx->d_feat_ring, (size_t)B * ctx->feat_rows * 96 * sizeof(float)));
    OWW_CUDA(ctx, cudaMalloc(&ctx->d_reset_ids, (size_t)B * sizeof(int)));
    OWW_CUDA(ctx, cudaMalloc(&ctx->d_reset_init, (size_t)ctx->feat_rows * 96 * sizeof(float)));
    ctx->n_streams = B;
    int rc = ensure_act(ctx, (size_t)std::min(B * mc, ctx->window_batch) * 74 * 32 * 24);
    if (rc) return rc;
    if ((rc = ensure_emb_tmp(ctx, (size_t)B * mc * 96))) return rc;
    if (ctx->cfg.cnn_mode == OWW_CNN_TC_INCREMENTAL && (rc = oww_late_alloc(ctx))) return rc;
    if (ctx->cfg.cnn_mode == OWW_CNN_TC_INCREMENTAL && (rc = oww_inc_alloc_streams(ctx))) return rc;
    return oww_reset(ctx, nullptr, B, nullptr, OWW_INIT_FEATURE_ROWS);
}

int oww_reset(oww_ctx* ctx, const int32_t* h_stream_ids, int n, const float* h_feature_init, int n_rows) {
    if (!ctx) return OWW_EINVAL;
    OWW_CUDA(ctx, cudaSetDevice(ctx->device));
    OWW_CUDA(ctx, cudaDeviceSynchronize());              // steps may be in flight on any stream
    int rc = reset_enqueue(ctx, h_stream_ids, n, h_feature_init, n_rows, nullptr);
    if (rc) return rc;
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return oww_fail(ctx, OWW_ECUDA, "reset failed: %s", cudaGetErrorString(e));
    return OWW_OK;
}

int oww_reset_async(oww_ctx* ctx, const int32_t* h_stream_ids, int n, const float* h_feature_init, int n_rows, void* stream) {
    if (!ctx) return OWW_EINVAL;
    OWW_CUDA(ctx, cudaSetDevice(ctx->device));
    return reset_enqueue(ctx, h_stream_ids, n, h_feature_init, n_rows, (cudaStream_t)stream);
}

int oww_step(oww_ctx* ctx, const int16_t* d_pcm, int64_t pcm_stride, int n_chunks, float* d_scores, void* stream) {
    if (!ctx || !d_pcm || !d_scores) return oww_fail(ctx, OWW_EINVAL, "null argument");
    OWW_CUDA(ctx, cudaSetDevice(ctx->device));
    return step_core(ctx, d_pcm, pcm_stride, n_chunks, d_scores, ctx->n_out_total, (cudaStream_t)stream);
}

int oww_step_host_submit(oww_ctx* ctx, const int16_t* h_pcm, int64_t pcm_stride, int n_chunks, int* ticket) {
    if (!ctx || !h_pcm || !ticket) return oww_fail(ctx, OWW_EINVAL, "null argument");
    OWW_CUDA(ctx, cudaSetDevice(ctx->device));
    const int B = ctx->n_streams;
    if (B <= 0) return oww_fail(ctx, OWW_EINVAL, "oww_set_streams has not been called");
    if (n_chunks < 1 || n_chunks > ctx->cfg.max_chunks)
        return oww_fail(ctx, OWW_EINVAL, "n_chunks=%d outside [1,%d]", n_chunks, ctx->cfg.max_chunks);
    const int si = ctx->next_slot;
    oww_ctx::HostSlot& S = ctx->slot[si];
    if (S.busy) return oww_fail(ctx, OWW_EINVAL, "both host slots are in flight: collect a ticket first");
    const size_t row = (size_t)n_chunks * OWW_SAMPLES_PER_CHUNK;
    const size_t pcm_bytes = (size_t)B * row * sizeof(int16_t);
    const size_t sc_bytes = (size_t)B * std::max(ctx->n_out_total, 1) * sizeof(float);
    if (!S.done) { OWW_CUDA(ctx, cudaEventCreateWithFlags(&S.done, cudaEventDisableTiming)); OWW_CUDA(ctx, cudaEventCreateWithFlags(&S.h2d_done, cudaEventDisableTiming)); }
    if (S.pcm_bytes < pcm_bytes) {
        cudaFreeHost(S.h_pcm); cudaFree(S.d_pcm); S.h_pcm = nullptr; S.d_pcm = nullptr; S.pcm_bytes = 0;
        OWW_CUDA(ctx, cudaMallocHost(&S.h_pcm, pcm_bytes));
        OWW_CUDA(ctx, cudaMalloc(&S.d_pcm, pcm_bytes));
        S.pcm_bytes = pcm_bytes;
    }
    if (S.sc_bytes < sc_bytes) {
        cudaFreeHost(S.h_scores); cudaFree(S.d_scores); S.h_scores = nullptr; S.d_scores = nullptr; S.sc_bytes = 0;
        OWW_CUDA(ctx, cudaMallocHost(&S.h_scores, sc_bytes));
        OWW_CUDA(ctx, cudaMalloc(&S.d_scores, sc_bytes));
        S.sc_bytes = sc_bytes;
    }
    // Source already page-locked (cudaMallocHost / cudaHostRegister / torch pin_memory) and dense: DMA straight from
    // the caller's buffer (it must stay untouched until the ticket is collected).  Otherwise stage through pinned memory.
    const int16_t* src = S.h_pcm;
    cudaPointerAttributes attr;
    const bool pinned = pcm_stride == (int64_t)row && cudaPointerGetAttributes(&attr, h_pcm) == cudaSuccess &&
                        attr.type == cudaMemoryTypeHost;
    cudaGetLastError();                                     // unregistered host memory reports an error on older drivers
    if (pinned) {
        src = h_pcm;
    } else if (pcm_stride == (int64_t)row) {
        std::memcpy(S.h_pcm, h_pcm, pcm_bytes);
    } else {
        for (int b = 0; b < B; ++b)
            std::memcpy(S.h_pcm + (size_t)b * row, h_pcm + (size_t)b * pcm_stride, row * sizeof(int16_t));
    }
    OWW_CUDA(ctx, cudaMemcpyAsync(S.d_pcm, src, pcm_bytes, cudaMemcpyHostToDevice, ctx->copy_stream));
    OWW_CUDA(ctx, cudaEventRecord(S.h2d_done, ctx->copy_stream));
    cudaStream_t s = ctx->own_stream;
    OWW_CUDA(ctx, cudaStreamWaitEvent(s, S.h2d_done, 0));
    int rc = step_core(ctx, S.d_pcm, (int64_t)row, n_chunks, S.d_scores, ctx->n_out_total, s);
    if (rc) return rc;
    if (ctx->n_out_total > 0)
        OWW_CUDA(ctx, cudaMemcpyAsync(S.h_scores, S.d_scores, (size_t)B * ctx->n_out_total * sizeof(float),
                                      cudaMemcpyDeviceToHost, s));
    OWW_CUDA(ctx, cudaEventRecord(S.done, s));
    S.busy = true;
    ctx->next_slot = si ^ 1;
    *ticket = si;
    return OWW_OK;
}

int oww_step_host_collect(oww_ctx* ctx, int ticket, float* h_scores) {
    if (!ctx || !h_scores) return oww_fail(ctx, OWW_EINVAL, "null argument");
    if (ticket < 0 || ticket > 1 || !ctx->slot[ticket].busy) return oww_fail(ctx, OWW_EINVAL, "ticket %d is not in flight", ticket);
    OWW_CUDA(ctx, cudaSetDevice(ctx->device));
    oww_ctx::HostSlot& S = ctx->slot[ticket];
    OWW_CUDA(ctx, cudaEventSynchronize(S.done));
    if (ctx->n_out_total > 0) std::memcpy(h_scores, S.h_scores, (size_t)ctx->n_streams * ctx->n_out_total * sizeof(float));
    S.busy = false;
    return OWW_OK;
}

int oww_step_host(oww_ctx* ctx, const int16_t* h_pcm, int64_t pcm_stride, int n_chunks, float* h_scores) {
    if (!ctx || !h_pcm || !h_scores) return oww_fail(ctx, OWW_EINVAL, "null argument");
    for (int i = 0; i < 2; ++i)
        if (ctx->slot[i].busy) return oww_fail(ctx, OWW_EINVAL, "a submitted step is still in flight: collect it first");
    int ticket = -1;
    int rc = oww_step_host_submit(ctx, h_pcm, pcm_stride, n_chunks, &ticket);
    if (rc) return rc;
    return oww_step_host_collect(ctx, ticket, h_scores);
}

int oww_get_features(oww_ctx* ctx, int stream_id, int n, int back, float* h_out) {
    if (!ctx || !h_out) return oww_fail(ctx, OWW_EINVAL, "null argument");
    if (stream_id < 0 || stream_id >= ctx->n_streams) return oww_fail(ctx, OWW_EINVAL, "bad stream id");
    if (n < 0 || back < 0 || n + back > ctx->feat_rows) return oww_fail(ctx, OWW_EINVAL, "n+back exceeds the ring (%d rows)", ctx->feat_rows);
    OWW_CUDA(ctx, cudaSetDevice(ctx->device));
    OWW_CUDA(ctx, cudaDeviceSynchronize());
    int count = 0;
    OWW_CUDA(ctx, cudaMemcpy(&count, ctx->d_feat_count + stream_id, sizeof(int), cudaMemcpyDeviceToHost));
    std::vector<float> ring((size_t)ctx->feat_rows * 96);
    OWW_CUDA(ctx, cudaMemcpy(ring.data(), ctx->d_feat_ring + (size_t)stream_id * ctx->feat_rows * 96,
                             ring.size() * sizeof(float), cudaMemcpyDeviceToHost));
    for (int i = 0; i < n; ++i) {
        const int r = count - back - n + i;
        if (r < 0 || r < count - ctx->feat_rows) std::memset(h_out + (size_t)i * 96, 0, 96 * sizeof(float));
        else std::memcpy(h_out + (size_t)i * 96, ring.data() + (size_t)(r & (ctx->feat_rows - 1)) * 96, 96 * sizeof(float));
    }
    return OWW_OK;
}

int oww_get_counts(oww_ctx* ctx, int stream_id, int* mel_rows, int* feature_rows) {
    if (!ctx) return OWW_EINVAL;
    if (stream_id < 0 || stream_id >= ctx->n_streams) return oww_fail(ctx, OWW_EINVAL, "bad stream id");
    OWW_CUDA(ctx, cudaSetDevice(ctx->device));
    OWW_CUDA(ctx, cudaDeviceSynchronize());
    int c[2] = {0, 0};
    OWW_CUDA(ctx, cudaMemcpy(&c[0], ctx->d_mel_count + stream_id, sizeof(int), cudaMemcpyDeviceToHost));
    OWW_CUDA(ctx, cudaMemcpy(&c[1], ctx->d_feat_count + stream_id, sizeof(int), cudaMemcpyDeviceToHost));
    if (mel_rows) *mel_rows = c[0];
    if (feature_rows) *feature_rows = c[1];
    return OWW_OK;
}

int oww_get_mel(oww_ctx* ctx, int stream_id, int n_rows, float* h_out) {
    if (!ctx || !h_out) return oww_fail(ctx, OWW_EINVAL, "null argument");
    if (stream_id < 0 || stream_id >= ctx->n_streams) return oww_fail(ctx, OWW_EINVAL, "bad stream id");
    if (n_rows < 0 || n_rows > OWW_WINDOW_ROWS) return oww_fail(ctx, OWW_EINVAL, "n_rows must be <= 76");
    OWW_CUDA(ctx, cudaSetDevice(ctx->device));
    OWW_CUDA(ctx, cudaDeviceSynchronize());
    int count = 0;
    OWW_CUDA(ctx, cudaMemcpy(&count, ctx->d_mel_count + stream_id, sizeof(int), cudaMemcpyDeviceToHost));
    std::vector<float> ring((size_t)ctx->mel_rows * 32);
    OWW_CUDA(ctx, cudaMemcpy(ring.data(), ctx->d_mel_ring + (size_t)stream_id * ctx->mel_rows * 32,
                             ring.size() * sizeof(float), cudaMemcpyDeviceToHost));
    for (int i = 0; i < n_rows; ++i) {
        const int r = count - n_rows + i;
        std::memcpy(h_out + (size_t)i * 32, ring.data() + (size_t)(r & (ctx->mel_rows - 1)) * 32, 32 * sizeof(float));
    }
    return OWW_OK;
}

int oww_embed_clips(oww_ctx* ctx, const int16_t* d_pcm, int n_clips, int n_samples, float* d_emb, void* stream) {
    if (!ctx || !d_pcm || !d_emb) return oww_fail(ctx, OWW_EINVAL, "null argument");
    if (n_samples < OWW_FFT_N) return oww_fail(ctx, OWW_EINVAL, "need at least 512 samples");
    OWW_CUDA(ctx, cudaSetDevice(ctx->device));
    const int T = (n_samples - OWW_FFT_N) / OWW_HOP + 1;
    if (T < OWW_WINDOW_ROWS)
        return oww_fail(ctx, OWW_EINVAL, "Embedding model requires the input melspectrograms to have at least 76 frames");
    const int W = (T - OWW_WINDOW_ROWS) / 8 + 1;
    cudaStream_t s = (cudaStream_t)stream;
    if (ctx->cfg.cnn_mode != OWW_CNN_FP32_WINDOW) {
        // tensor-core modes: per-clip mel (one call per clip, as the reference's CPU path runs the graph), then ONE fully
        // convolutional tcgen05 pass over the clip's [T x 32] mel (SURVEY.md F10) - slabs bounded by a ~1 GB plane scratch
        const int t_use = OWW_WINDOW_ROWS + 8 * (W - 1);
        const size_t per1 = oww_tc_act_units_T(ctx, 1, t_use);
        int slab = (int)std::max<size_t>(1, ((size_t)1 << 26) / per1);          // 2^26 units = 1 GiB per buffer
        slab = std::min(slab, n_clips);
        int rc = ensure_tc_units(ctx, oww_tc_act_units_T(ctx, slab, t_use));
        if (rc) return rc;
        float* d_mel = nullptr;
        OWW_CUDA(ctx, cudaMallocAsync(&d_mel, (size_t)slab * T * 32 * sizeof(float), s));
        for (int c0 = 0; c0 < n_clips; c0 += slab) {
            const int m = std::min(slab, n_clips - c0);
            MelLaunch ml{d_pcm + (size_t)c0 * n_samples, (int64_t)n_samples, n_samples, nullptr, nullptr, d_mel, (int64_t)T * 32,
                         -1, nullptr, m, 1, 0};
            if ((rc = oww_mel_launch(ctx, ml, s))) break;
            if ((rc = oww_cnn_tc_clip(ctx, d_mel, m, T, d_emb + (size_t)c0 * W * 96, s))) break;
        }
        cudaFreeAsync(d_mel, s);
        return rc;
    }
    // slabs bounded by the activation scratch (~512 windows' worth of layer-1 output)
    const size_t per_clip = (size_t)(T - 2) * 32 * 24;
    int rc = ensure_act(ctx, std::max(ctx->act_floats, std::max(per_clip, (size_t)ctx->window_batch * 74 * 32 * 24)));
    if (rc) return rc;
    const int slab = (int)std::max<size_t>(1, ctx->act_floats / per_clip);
    float* d_mel = nullptr;
    OWW_CUDA(ctx, cudaMallocAsync(&d_mel, (size_t)std::min(slab, n_clips) * T * 32 * sizeof(float), s));
    for (int c0 = 0; c0 < n_clips; c0 += slab) {
        const int m = std::min(slab, n_clips - c0);
        MelLaunch ml{d_pcm + (size_t)c0 * n_samples, (int64_t)n_samples, n_samples, nullptr, nullptr, d_mel, (int64_t)T * 32,
                     -1, nullptr, m, 1, 0};
        if ((rc = oww_mel_launch(ctx, ml, s))) break;
        if ((rc = oww_cnn_clip_fp32(ctx, d_mel, m, T, d_emb + (size_t)c0 * W * 96, s))) break;
    }
    cudaFreeAsync(d_mel, s);
    return rc;
}

int oww_predict_clips(oww_ctx* ctx, const int16_t* d_pcm, int n_clips, int n_samples, int pad_samples,
                      const float* h_feature_init, int n_rows, float* d_scores, void* stream) {
    if (!ctx || !d_pcm || !d_scores) return oww_fail(ctx, OWW_EINVAL, "null argument");
    if (n_clips < 1 || n_samples < 1 || pad_samples < 0) return oww_fail(ctx, OWW_EINVAL, "bad clip geometry");
    OWW_CUDA(ctx, cudaSetDevice(ctx->device));
    const int64_t L = (int64_t)n_samples + 2 * (int64_t)pad_samples;
    const int steps = L > OWW_SAMPLES_PER_CHUNK ? (int)((L - OWW_SAMPLES_PER_CHUNK + OWW_SAMPLES_PER_CHUNK - 1) / OWW_SAMPLES_PER_CHUNK) : 0;
    if (steps == 0) return OWW_OK;
    cudaStream_t s = (cudaStream_t)stream;
    {
        // ---- bulk path (SURVEY.md F10): per slab of clips ONE mel launch over the padded clips (frames grouped and
        //      clamped per streaming call, behind the 71 rows of ones a fresh stream's window starts with), ONE fully
        //      convolutional tcgen05 pass per conv layer over [76 + 8 (steps-1)] x 32, then the heads over all sliding
        //      windows of [feature_init rows | embeddings] in one launch.  Bit-identical to streaming the clips.
        bool tc_all = ctx->cfg.cnn_mode != OWW_CNN_FP32_WINDOW && steps <= 8192 && !ctx->heads.empty();
        for (size_t i = 0; i < ctx->heads.size(); ++i) tc_all = tc_all && oww_heads_tc_supported(ctx, (int)i);
        if (tc_all) {
            const int T_v = OWW_WINDOW_ROWS + 8 * (steps - 1);
            const int init_rows = h_feature_init ? n_rows : OWW_INIT_FEATURE_ROWS;
            const int64_t f_stride = (int64_t)(init_rows + steps) * 96;
            const size_t per1 = oww_tc_act_units_T(ctx, 1, T_v);
            int slab = (int)std::max<size_t>(1, ((size_t)1 << 26) / per1);      // 1 GiB of fp16 planes per buffer
            slab = std::min(slab, n_clips);
            int rc = ensure_tc_units(ctx, oww_tc_act_units_T(ctx, slab, T_v));
            if (rc) return rc;
            float *d_v = nullptr, *d_f = nullptr, *d_init = nullptr;
            OWW_CUDA(ctx, cudaMallocAsync(&d_v, (size_t)slab * T_v * 32 * sizeof(float), s));
            OWW_CUDA(ctx, cudaMallocAsync(&d_f, (size_t)slab * f_stride * sizeof(float), s));
            if (h_feature_init && init_rows > 0) {
                OWW_CUDA(ctx, cudaMallocAsync(&d_init, (size_t)init_rows * 96 * sizeof(float), s));
                OWW_CUDA(ctx, cudaMemcpyAsync(d_init, h_feature_init, (size_t)init_rows * 96 * sizeof(float), cudaMemcpyHostToDevice, s));
            }
            for (int c0 = 0; c0 < n_clips && rc == OWW_OK; c0 += slab) {
                const int m = std::min(slab, n_clips - c0);
                if ((rc = oww_mel_clips_launch(ctx, d_pcm + (size_t)c0 * n_samples, n_samples, m, n_samples, pad_samples, steps, d_v,
                                               (int64_t)T_v * 32, s))) break;
                if (init_rows > 0) {
                    fill_init_rows_kernel<<<std::min(1024, (m * init_rows * 24 + 255) / 256), 256, 0, s>>>(d_f, f_stride, m, d_init, init_rows);
                    ctx->launches++;
                }
                // embeddings of step st land at row init_rows + st of the clip's feature array
                WindowSrc src{d_v, (int64_t)T_v * 32, nullptr, -1, 0, 0};
                if ((rc = oww_cnn_tc_clip_rows(ctx, src, m, T_v, d_f + (int64_t)init_rows * 96, init_rows + steps, s))) break;
                FeatSrc fs{d_f, f_stride, nullptr, -1, 0};
                fs.steps = steps; fs.row0 = init_rows;
                rc = oww_heads_all(ctx, fs, m * steps, d_scores + (size_t)c0 * steps * ctx->n_out_total, ctx->n_out_total, 0, s);
            }
            cudaFreeAsync(d_v, s); cudaFreeAsync(d_f, s);
            if (d_init) cudaFreeAsync(d_init, s);
            return rc;
        }
    }
    const int slab_max = 16384;
    // the private stream set shares this handle's weights (shallow copy, non-owning)
    if (!ctx->clip_ctx) {
        oww_ctx* c = new (std::nothrow) oww_ctx();
        if (!c) return oww_fail(ctx, OWW_ENOMEM, "out of host memory");
        c->cfg = ctx->cfg; c->cfg.max_chunks = 1; c->device = ctx->device; c->sm_count = ctx->sm_count;
        c->window_batch = ctx->window_batch;
        c->fuse_step = ctx->fuse_step; c->tc_heads = ctx->tc_heads; c->tc_heads_terms = ctx->tc_heads_terms;
        cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking);
        ctx->clip_ctx = c;
    }
    oww_ctx* c = ctx->clip_ctx;
    c->mel_loaded = ctx->mel_loaded; c->d_window = ctx->d_window; c->d_twiddle = ctx->d_twiddle;
    c->d_mel_start = ctx->d_mel_start; c->d_mel_len = ctx->d_mel_len; c->d_mel_w = ctx->d_mel_w; c->mel_kmax = ctx->mel_kmax;
    if (c->emb_loaded != ctx->emb_loaded || c->d_inc_w != ctx->d_inc_w) c->tails_template_valid = false;
    c->emb_loaded = ctx->emb_loaded;
    for (int li = 0; li < OWW_N_CONV; ++li) { c->conv[li] = ctx->conv[li]; c->tc_w_off[li] = ctx->tc_w_off[li]; c->tc_sb_off[li] = ctx->tc_sb_off[li]; }
    c->d_tc_w = ctx->d_tc_w; c->d_tc_sb = ctx->d_tc_sb; c->d_inc_w = ctx->d_inc_w;
    c->d_tc_w3 = ctx->d_tc_w3; c->d_tc_sb3 = ctx->d_tc_sb3; c->split_from = ctx->split_from;

    c->heads = ctx->heads; c->n_out_total = ctx->n_out_total; c->max_n_in = ctx->max_n_in; c->d_head_devs = ctx->d_head_devs;
    c->gates = ctx->gates; c->d_gates = ctx->d_gates;
    int rc = OWW_OK;
    for (int c0 = 0; c0 < n_clips && rc == OWW_OK; c0 += slab_max) {
        const int m = std::min(slab_max, n_clips - c0);
        if (c->n_streams != m) { if ((rc = oww_set_streams(c, m))) { ctx->err = c->err; break; } }
        if ((rc = oww_reset(c, nullptr, m, h_feature_init, h_feature_init ? n_rows : OWW_INIT_FEATURE_ROWS))) { ctx->err = c->err; break; }
        const size_t stage_bytes = (size_t)m * OWW_SAMPLES_PER_CHUNK * sizeof(int16_t);
        if (c->slot[0].pcm_bytes < stage_bytes) {
            cudaFree(c->slot[0].d_pcm); c->slot[0].d_pcm = nullptr;
            OWW_CUDA(ctx, cudaMalloc(&c->slot[0].d_pcm, stage_bytes));
            c->slot[0].pcm_bytes = stage_bytes;
        }
        for (int st = 0; st < steps; ++st) {
            unsigned grid = (unsigned)std::min<int64_t>(((int64_t)m * OWW_SAMPLES_PER_CHUNK + 255) / 256, (int64_t)ctx->sm_count * 32);
            gather_chunk_kernel<<<grid, 256, 0, s>>>(d_pcm + (size_t)c0 * n_samples, m, n_samples, pad_samples, st, c->slot[0].d_pcm);
            c->launches++;
            rc = step_core(c, c->slot[0].d_pcm, OWW_SAMPLES_PER_CHUNK, 1,
                           d_scores + ((size_t)c0 * steps + st) * ctx->n_out_total, steps * ctx->n_out_total, s);
            if (rc) { ctx->err = c->err; break; }
        }
    }
    ctx->launches += c->launches; c->launches = 0;
    c->heads.clear();   // do not let the child free shared blobs
    c->d_head_devs = nullptr;
    c->gates.clear(); c->d_gates = nullptr;
    return rc;
}

int oww_debug_layer(oww_ctx* ctx, const float* d_windows, int n, int layer, float* d_out, void* stream) {
    if (!ctx || !d_windows || !d_out) return oww_fail(ctx, OWW_EINVAL, "null argument");
    if (layer < 0 || layer >= OWW_N_CONV - 1) return oww_fail(ctx, OWW_EINVAL, "layer must be in [0,18]");
    if (n < 1 || n > ctx->window_batch) return oww_fail(ctx, OWW_EINVAL, "n must be in [1, window_batch]");
    OWW_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = ensure_act(ctx, (size_t)std::min(n, ctx->window_batch) * 74 * 32 * 24);
    if (rc) return rc;
    WindowSrc src{d_windows, (int64_t)OWW_WINDOW_ROWS * 32, nullptr, -1, 0, 0};
    if (ctx->cfg.cnn_mode == OWW_CNN_TC_WINDOW) return oww_cnn_tc_pyramid(ctx, src, n, nullptr, layer, d_out, (cudaStream_t)stream);
    return oww_cnn_fp32_pyramid(ctx, src, n, nullptr, layer, d_out, (cudaStream_t)stream);
}

int oww_debug_inc_plan(oww_ctx* ctx, int group, int n_streams, int32_t* out, int max_ints) {
    if (!out) return oww_fail(ctx, OWW_EINVAL, "null argument");
    oww_ctx local;                       // ctx may be NULL: the plan depends only on the fixed layer table
    if (!ctx) { fill_layer_table(&local); ctx = &local; }
    IncPlan P;
    int rc = oww_inc_build_plan(ctx, group, n_streams, OWW_N_CONV, &P);
    if (rc) return rc;
    const int n = (int)(sizeof(IncPlan) / sizeof(int32_t));
    if (max_ints < n) return oww_fail(ctx, OWW_EINVAL, "need room for %d ints", n);
    std::memcpy(out, &P, sizeof(IncPlan));
    return n;
}

int oww_debug_inc_clocks(oww_ctx* ctx, int64_t* h_out21) {
    if (!ctx || !h_out21) return oww_fail(ctx, OWW_EINVAL, "null argument");
    if (ctx->cfg.cnn_mode != OWW_CNN_TC_INCREMENTAL || ctx->n_streams <= 0)
        return oww_fail(ctx, OWW_EINVAL, "needs cnn_mode 3 with streams allocated");
    OWW_CUDA(ctx, cudaSetDevice(ctx->device));
    OWW_CUDA(ctx, cudaDeviceSynchronize());
    if (!ctx->d_inc_dbg) OWW_CUDA(ctx, cudaMalloc(&ctx->d_inc_dbg, 104 * sizeof(int64_t)));
    OWW_CUDA(ctx, cudaMemset(ctx->d_inc_dbg, 0, 104 * sizeof(int64_t)));
    // stamps are taken by the NEXT step the caller runs; this call only arms the buffer
    return OWW_OK;
}

int oww_debug_inc_clocks_read(oww_ctx* ctx, int64_t* h_out21) {
    if (!ctx || !h_out21 || !ctx->d_inc_dbg) return oww_fail(ctx, OWW_EINVAL, "clock buffer not armed");
    OWW_CUDA(ctx, cudaSetDevice(ctx->device));
    OWW_CUDA(ctx, cudaDeviceSynchronize());
    OWW_CUDA(ctx, cudaMemcpy(h_out21, ctx->d_inc_dbg, 104 * sizeof(int64_t), cudaMemcpyDeviceToHost));
    cudaFree(ctx->d_inc_dbg); ctx->d_inc_dbg = nullptr;
    return OWW_OK;
}

int oww_enable_stage_timing(oww_ctx* ctx, int n_slots) {
    if (!ctx) return OWW_EINVAL;
    OWW_CUDA(ctx, cudaSetDevice(ctx->device));
    ctx->timing = n_slots > 0;
    ctx->ev_steps = 0;
    if (n_slots > 4096) n_slots = 4096;
    while ((int)ctx->ev.size() < 4 * n_slots) {
        cudaEvent_t e;
        OWW_CUDA(ctx, cudaEventCreate(&e));
        ctx->ev.push_back(e);
    }
    if (n_slots > 0) { ctx->ev_slots = n_slots; ctx->ev_fused.assign(n_slots, 0); }
    return OWW_OK;
}

int oww_stage_ms(oww_ctx* ctx, float out_ms[3]) {
    if (!ctx || !out_ms) return OWW_EINVAL;
    if (!ctx->timing || ctx->ev_steps == 0) return oww_fail(ctx, OWW_EINVAL, "no timed step recorded");
    const long n = ctx->ev_steps < ctx->ev_slots ? ctx->ev_steps : ctx->ev_slots;
    double acc[3] = {0, 0, 0};
    for (long k = 0; k < n; ++k) {
        cudaEvent_t* ev = &ctx->ev[4 * k];
        // 0: mel | cnn | heads launches (events 0..3)   1: one fused launch (events 1..2)
        // 2: fused frontend+CNN launch, then a heads launch (events 1..3)
        const int kind = ctx->ev_fused[k];
        const int first = kind == 0 ? 0 : 1, last = kind == 1 ? 2 : 3;
        OWW_CUDA(ctx, cudaEventSynchronize(ev[last]));
        for (int i = first; i < last; ++i) {
            float ms = 0.f;
            OWW_CUDA(ctx, cudaEventElapsedTime(&ms, ev[i], ev[i + 1]));
            acc[i] += ms;
        }
    }
    for (int i = 0; i < 3; ++i) out_ms[i] = (float)(acc[i] / n);
    return OWW_OK;
}

}  // extern "C"
