// nnj_api.cu — the C ABI declared in include/nnj.h.
#include <cstdio>
#include <cstring>
#include <new>

#include <cuda_bf16.h>

#include "nnj_internal.h"

namespace nnj {

thread_local long long g_launches = 0;
static thread_local char g_err[512] = "";

int set_error(int code, const char* msg) {
    snprintf(g_err, sizeof(g_err), "%s", msg);
    return code;
}

int set_cuda_error(cudaError_t e, const char* file, int line) {
    snprintf(g_err, sizeof(g_err), "CUDA error %d (%s) at %s:%d", (int)e, cudaGetErrorString(e), file, line);
    return NNJ_ERR_CUDA;
}

int current_device() {
    int dev = 0;
    cudaGetDevice(&dev);
    return dev;
}

int sm_count() {
    static std::atomic<int> cache[64];
    const int dev = current_device() & 63;
    int n = cache[dev].load(std::memory_order_relaxed);
    if (n <= 0) {
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cache[dev].store(n, std::memory_order_relaxed);
    }
    return n;
}

// ---- optional per-kernel-class timing with CUDA events on the launching stream ----
struct ProfRec { int cls; cudaEvent_t a, b; };
static thread_local bool g_prof_on = false;
static thread_local std::vector<ProfRec> g_prof;
static thread_local std::vector<cudaEvent_t> g_prof_pool;
static thread_local int g_prof_open = -1;

static cudaEvent_t prof_event() {
    if (!g_prof_pool.empty()) { cudaEvent_t e = g_prof_pool.back(); g_prof_pool.pop_back(); return e; }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}

void prof_begin(int cls, cudaStream_t st) {
    if (!g_prof_on) return;
    ProfRec r{cls, prof_event(), prof_event()};
    cudaEventRecord(r.a, st);
    g_prof.push_back(r);
    g_prof_open = (int)g_prof.size() - 1;
}

void prof_end(cudaStream_t st) {
    if (!g_prof_on || g_prof_open < 0) return;
    cudaEventRecord(g_prof[g_prof_open].b, st);
    g_prof_open = -1;
}

static const char* kclass_names[KC_COUNT] = {"embed", "ln_qkv", "row_qk_gemm", "row_softmax", "row_pv_gemm", "out_proj", "col_attn",
                                             "ffn", "node_derive", "alpha", "alpha_softmax", "pair_score", "select", "merge", "misc", "pair_blend", "tree_llh"};

#define CUDA_TRY(x)                                                        \
    do {                                                                   \
        cudaError_t e_ = (x);                                              \
        if (e_ != cudaSuccess) return set_cuda_error(e_, __FILE__, __LINE__); \
    } while (0)

// host-side packing helpers -------------------------------------------------
struct Packer {
    std::vector<float> host;
    size_t add(const float* p, size_t n) {          // plain copy, 16-byte aligned start
        size_t off = (host.size() + 3) / 4 * 4;
        host.resize(off + n);
        memcpy(host.data() + off, p, n * sizeof(float));
        return off;
    }
    size_t add_t(const float* w, int out, int in) { // W [out][in] -> Wt [in][out]
        size_t off = (host.size() + 3) / 4 * 4;
        host.resize(off + (size_t)out * in);
        for (int o = 0; o < out; ++o)
            for (int i = 0; i < in; ++i) host[off + (size_t)i * out + o] = w[(size_t)o * in + i];
        return off;
    }
};

}  // namespace nnj

using namespace nnj;

struct nnj_model : public nnj::Model {};

extern "C" {

const char* nnj_last_error(void) { return g_err; }
int nnj_abi_version(void) { return NNJ_ABI_VERSION; }

int nnj_profile_enable(int on) {
    for (auto& r : g_prof) { g_prof_pool.push_back(r.a); g_prof_pool.push_back(r.b); }
    g_prof.clear();
    g_prof_open = -1;
    g_prof_on = on != 0;
    return NNJ_OK;
}

int nnj_profile_classes(void) { return KC_COUNT; }

const char* nnj_profile_name(int cls) { return (cls >= 0 && cls < KC_COUNT) ? kclass_names[cls] : ""; }

int nnj_profile_read(int n, double* ms, int64_t* launches) {
    if (n < KC_COUNT || !ms || !launches) return set_error(NNJ_ERR_INVALID, "profile_read: need room for nnj_profile_classes() entries");
    for (int i = 0; i < n; ++i) { ms[i] = 0.0; launches[i] = 0; }
    CUDA_TRY(cudaDeviceSynchronize());
    for (auto& r : g_prof) {
        float t = 0.f;
        if (cudaEventElapsedTime(&t, r.a, r.b) == cudaSuccess) { ms[r.cls] += t; launches[r.cls] += 1; }
    }
    return NNJ_OK;
}

int64_t nnj_launch_count(int reset) {
    long long v = g_launches;
    if (reset) g_launches = 0;
    return v;
}

int nnj_model_create(nnj_model** out, const nnj_config* cfg, const float* const* tensors, const int64_t* numels, int n_tensors,
                     int device) {
    if (!out || !cfg || !tensors || !numels) return set_error(NNJ_ERR_INVALID, "model_create: null argument");
    if (cfg->embed_dim != 64 || cfg->num_heads != 8 || cfg->vocab_size != 4 || cfg->patch_size != 1 || cfg->num_layers < 1)
        return set_error(NNJ_ERR_INVALID,
                         "model_create: unsupported config (need embed_dim 64, num_heads 8, vocab_size 4, patch_size 1, num_layers >= 1)");
    if (cfg->precision != NNJ_PREC_FP32 && cfg->precision != NNJ_PREC_BF16X3 && cfg->precision != NNJ_PREC_BF16)
        return set_error(NNJ_ERR_INVALID, "model_create: unknown precision mode");
    const int Lyr = cfg->num_layers;
    if (n_tensors != Lyr * 26 + 16) return set_error(NNJ_ERR_INVALID, "model_create: expected 26 tensors per layer + 16");
    // expected element counts in state_dict order
    std::vector<int64_t> expect;
    for (int l = 0; l < Lyr; ++l) {
        for (int blk = 0; blk < 2; ++blk) {
            for (int p = 0; p < 4; ++p) { expect.push_back(64 * 64); expect.push_back(64); }
            expect.push_back(64); expect.push_back(64);
        }
        expect.push_back(256 * 64); expect.push_back(256); expect.push_back(64 * 256); expect.push_back(64);
        expect.push_back(64); expect.push_back(64);
    }
    const int64_t tail[16] = {64 * 4, 64, 64 * 64, 64, 64 * 64, 64, 64 * 64, 64, 64 * 64, 64, 64 * 64, 64, 64 * 64, 64, 64, 1};
    for (int i = 0; i < 16; ++i) expect.push_back(tail[i]);
    for (int i = 0; i < n_tensors; ++i)
        if (numels[i] != expect[i]) {
            char msg[128];
            snprintf(msg, sizeof(msg), "model_create: tensor %d has %lld elements, expected %lld", i, (long long)numels[i], (long long)expect[i]);
            return set_error(NNJ_ERR_INVALID, msg);
        }
    DeviceGuard guard(device);              // the caller's current device (PyTorch's) is restored on return
    if (guard.err != cudaSuccess) return set_cuda_error(guard.err, __FILE__, __LINE__);
    nnj_model* m = new (std::nothrow) nnj_model();
    if (!m) return set_error(NNJ_ERR_NOMEM, "model_create: out of host memory");
    m->cfg = *cfg; m->device = device; m->num_layers = Lyr; m->blob = nullptr; m->blob_bf = nullptr; m->blob_enc = nullptr; m->host_ws = nullptr; m->host_ws_bytes = 0;
    m->host_compute = nullptr; m->host_copy = nullptr;

    Packer pk;
    struct AttnOff { size_t ln_g, ln_b, qt, kt, vt, ot, qb, kb, vb, ob, qkvb; };
    struct LayerOff { AttnOff a[2]; size_t fln_g, fln_b, w1t, b1, w2t, b2; };
    std::vector<LayerOff> lo(Lyr);
    int ti = 0;
    for (int l = 0; l < Lyr; ++l) {
        for (int blk = 0; blk < 2; ++blk) {
            AttnOff& a = lo[l].a[blk];
            // state_dict order: k_proj, v_proj, q_proj, out_proj (axial_attention.py:24-28), then the block's LayerNorm
            a.kt = pk.add_t(tensors[ti], 64, 64); a.kb = pk.add(tensors[ti + 1], 64);
            a.vt = pk.add_t(tensors[ti + 2], 64, 64); a.vb = pk.add(tensors[ti + 3], 64);
            a.qt = pk.add_t(tensors[ti + 4], 64, 64); a.qb = pk.add(tensors[ti + 5], 64);
            a.ot = pk.add_t(tensors[ti + 6], 64, 64); a.ob = pk.add(tensors[ti + 7], 64);
            a.ln_g = pk.add(tensors[ti + 8], 64); a.ln_b = pk.add(tensors[ti + 9], 64);
            a.qkvb = pk.add(tensors[ti + 5], 64); pk.add(tensors[ti + 1], 64); pk.add(tensors[ti + 3], 64);   // q|k|v biases, contiguous
            ti += 10;
        }
        // fc1 [256][64] -> 4 chunks of [64 k][64 col]; fc2 [64][256] -> 4 chunks of [64 hidden][64 out]
        {
            const float* w1 = tensors[ti];
            std::vector<float> t1(4 * 4096), t2(4 * 4096);
            for (int ch = 0; ch < 4; ++ch)
                for (int k = 0; k < 64; ++k)
                    for (int c = 0; c < 64; ++c) t1[ch * 4096 + k * 64 + c] = w1[(size_t)(ch * 64 + c) * 64 + k];
            const float* w2 = tensors[ti + 2];
            for (int ch = 0; ch < 4; ++ch)
                for (int k = 0; k < 64; ++k)
                    for (int o = 0; o < 64; ++o) t2[ch * 4096 + k * 64 + o] = w2[(size_t)o * 256 + ch * 64 + k];
            lo[l].w1t = pk.add(t1.data(), t1.size()); lo[l].b1 = pk.add(tensors[ti + 1], 256);
            lo[l].w2t = pk.add(t2.data(), t2.size()); lo[l].b2 = pk.add(tensors[ti + 3], 64);
            lo[l].fln_g = pk.add(tensors[ti + 4], 64); lo[l].fln_b = pk.add(tensors[ti + 5], 64);
            ti += 6;
        }
    }
    size_t e_w1 = pk.add(tensors[ti], 256), e_b1 = pk.add(tensors[ti + 1], 64);
    size_t e_w2t = pk.add_t(tensors[ti + 2], 64, 64), e_b2 = pk.add(tensors[ti + 3], 64);
    size_t h_t = pk.add_t(tensors[ti + 4], 64, 64), h_b = pk.add(tensors[ti + 5], 64);
    size_t g_t = pk.add_t(tensors[ti + 6], 64, 64), g_b = pk.add(tensors[ti + 7], 64);
    size_t q_w = pk.add(tensors[ti + 8], 4096), q_b = pk.add(tensors[ti + 9], 64);
    size_t k_t = pk.add_t(tensors[ti + 10], 64, 64), k_b = pk.add(tensors[ti + 11], 64);
    size_t s_t = pk.add_t(tensors[ti + 12], 64, 64), s_b = pk.add(tensors[ti + 13], 64);
    size_t s2_w = pk.add(tensors[ti + 14], 64);
    const float s2_b = tensors[ti + 15][0];

    cudaError_t e = cudaMalloc(&m->blob, pk.host.size() * sizeof(float));
    if (e != cudaSuccess) { delete m; return set_cuda_error(e, __FILE__, __LINE__); }
    e = cudaMemcpy(m->blob, pk.host.data(), pk.host.size() * sizeof(float), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { cudaFree(m->blob); delete m; return set_cuda_error(e, __FILE__, __LINE__); }
    const float* B0 = m->blob;
    m->layers.resize(Lyr);
    for (int l = 0; l < Lyr; ++l) {
        AttnW* aw[2] = {&m->layers[l].row, &m->layers[l].col};
        for (int blk = 0; blk < 2; ++blk) {
            const AttnOff& a = lo[l].a[blk];
            *aw[blk] = AttnW{B0 + a.ln_g, B0 + a.ln_b, B0 + a.qt, B0 + a.kt, B0 + a.vt, B0 + a.ot, B0 + a.qb, B0 + a.kb, B0 + a.vb, B0 + a.ob};
        }
        m->layers[l].ffn = FfnW{B0 + lo[l].fln_g, B0 + lo[l].fln_b, B0 + lo[l].w1t, B0 + lo[l].b1, B0 + lo[l].w2t, B0 + lo[l].b2};
    }
    m->embed = EmbedW{B0 + e_w1, B0 + e_b1, B0 + e_w2t, B0 + e_b2};
    m->nj = NjW{B0 + h_t, B0 + h_b, B0 + g_t, B0 + g_b, B0 + q_w, B0 + q_b, B0 + k_t, B0 + k_b, B0 + s_t, B0 + s_b, B0 + s2_w, s2_b};
    {   // bf16 hi/lo planes of the two [64][64] weights used as K-major B operands by the tensor-core pair-score kernel
        std::vector<uint16_t> planes(4 * 4096 + 4 * 8192);
        const float* src[2] = {tensors[ti + 6] /*g_linear_last*/, tensors[ti + 12] /*s_out.0*/};
        {   // mma.sync B fragments (NjFrag) of the merge / node-derive weights: B[k][n] = W[n][k] for the torch Linear weights, Wq as it is
            const float* wsrc[4] = {tensors[ti + 4] /*h_linear_last*/, tensors[ti + 10] /*g_attn_k*/, tensors[ti + 8] /*g_attn_q*/, tensors[ti + 6] /*g_linear_last*/};
            const bool transposed[4] = {true, true, false, true};
            for (int w = 0; w < 4; ++w) {
                uint16_t* out = planes.data() + 4 * 4096 + (size_t)w * 8192;
                auto Bm = [&](int k, int n) { return transposed[w] ? wsrc[w][n * 64 + k] : wsrc[w][k * 64 + n]; };
                for (int ks = 0; ks < 4; ++ks)
                    for (int nt = 0; nt < 8; ++nt)
                        for (int lane = 0; lane < 32; ++lane) {
                            const int g = lane >> 2, t = lane & 3, n = nt * 8 + g;
                            const int kk[4] = {ks * 16 + 2 * t, ks * 16 + 2 * t + 1, ks * 16 + 2 * t + 8, ks * 16 + 2 * t + 9};
                            uint16_t* e = out + ((size_t)(ks * 8 + nt) * 32 + lane) * 8;
                            for (int i = 0; i < 4; ++i) {
                                const float v = Bm(kk[i], n);
                                const __nv_bfloat16 h = __float2bfloat16_rn(v);
                                const __nv_bfloat16 l = NNJ_LO_BF16(__float2bfloat16_rn(v - __bfloat162float(h)));
                                e[i] = __bfloat16_as_ushort(h);
                                e[4 + i] = __bfloat16_as_ushort(l);
                            }
                        }
            }
        }
        for (int w = 0; w < 2; ++w)
            for (int i = 0; i < 4096; ++i) {
                __nv_bfloat16 h = __float2bfloat16_rn(src[w][i]);
                __nv_bfloat16 l = NNJ_LO_BF16(__float2bfloat16_rn(src[w][i] - __bfloat162float(h)));
                planes[(2 * w) * 4096 + i] = __bfloat16_as_ushort(h);
                planes[(2 * w + 1) * 4096 + i] = __bfloat16_as_ushort(l);
            }
        e = cudaMalloc(&m->blob_bf, planes.size() * 2);
        if (e == cudaSuccess) e = cudaMemcpy(m->blob_bf, planes.data(), planes.size() * 2, cudaMemcpyHostToDevice);
        if (e != cudaSuccess) { cudaFree(m->blob); if (m->blob_bf) cudaFree(m->blob_bf); delete m; return set_cuda_error(e, __FILE__, __LINE__); }
        const uint16_t* pb = reinterpret_cast<const uint16_t*>(m->blob_bf);
        m->nj_bf = NjBf{pb, pb + 4096, pb + 8192, pb + 12288};
        const uint4* pf = reinterpret_cast<const uint4*>(pb + 4 * 4096);
        m->nj_frag = NjFrag{pf, pf + 1024, pf + 2048, pf + 3072};
    }
    {   // shared-memory images of the encoder weights for the tcgen05 kernels (EncTcW)
        constexpr size_t QKV = 2 * 192 * 64, OW = 2 * 64 * 64, W1 = 2 * 256 * 64, W2 = 2 * 64 * 256;   // bf16 elements
        constexpr size_t PER = 2 * QKV + 2 * OW + W1 + W2;
        std::vector<uint16_t> img((size_t)Lyr * PER, 0);
        // W [N][ldw] rows n, K window [k0, k0+64) -> [N][64] K-major SWIZZLE_128B image, hi plane at dst_h, lo plane at dst_l
        auto put = [&](uint16_t* dst_h, uint16_t* dst_l, const float* W, int n_rows, int ldw, int k0, int row0) {
            for (int n = 0; n < n_rows; ++n)
                for (int k = 0; k < 64; ++k) {
                    const float v = W[(size_t)n * ldw + k0 + k];
                    const __nv_bfloat16 h = __float2bfloat16_rn(v), l = NNJ_LO_BF16(__float2bfloat16_rn(v - __bfloat162float(h)));
                    const int rn = row0 + n;
                    const size_t off = (size_t)rn * 64 + (size_t)(((k >> 3) ^ (rn & 7)) << 3) + (k & 7);
                    dst_h[off] = __bfloat16_as_ushort(h);
                    dst_l[off] = __bfloat16_as_ushort(l);
                }
        };
        int tj = 0;
        for (int l = 0; l < Lyr; ++l) {
            uint16_t* base = img.data() + (size_t)l * PER;
            uint16_t* qkv[2] = {base, base + QKV + OW};
            uint16_t* ow[2] = {base + QKV, base + 2 * QKV + OW};
            for (int blk = 0; blk < 2; ++blk) {   // state_dict order: k_proj, v_proj, q_proj, out_proj
                put(qkv[blk], qkv[blk] + 192 * 64, tensors[tj + 4], 64, 64, 0, 0);     // q rows 0..63
                put(qkv[blk], qkv[blk] + 192 * 64, tensors[tj + 0], 64, 64, 0, 64);    // k rows 64..127
                put(qkv[blk], qkv[blk] + 192 * 64, tensors[tj + 2], 64, 64, 0, 128);   // v rows 128..191
                put(ow[blk], ow[blk] + 64 * 64, tensors[tj + 6], 64, 64, 0, 0);
                tj += 10;
            }
            uint16_t* w1 = base + 2 * QKV + 2 * OW;
            uint16_t* w2 = w1 + W1;
            put(w1, w1 + 256 * 64, tensors[tj], 256, 64, 0, 0);
            for (int kc = 0; kc < 4; ++kc) put(w2 + (size_t)kc * 4096, w2 + 64 * 256 + (size_t)kc * 4096, tensors[tj + 2], 64, 256, kc * 64, 0);
            tj += 6;
        }
        e = cudaMalloc(&m->blob_enc, img.size() * 2);
        if (e == cudaSuccess) e = cudaMemcpy(m->blob_enc, img.data(), img.size() * 2, cudaMemcpyHostToDevice);
        if (e != cudaSuccess) { cudaFree(m->blob); cudaFree(m->blob_bf); if (m->blob_enc) cudaFree(m->blob_enc); delete m; return set_cuda_error(e, __FILE__, __LINE__); }
        const uint16_t* pe = reinterpret_cast<const uint16_t*>(m->blob_enc);
        m->enc_tc.resize(Lyr);
        for (int l = 0; l < Lyr; ++l) {
            const uint16_t* base = pe + (size_t)l * PER;
            EncTcW& w = m->enc_tc[l];
            w.row_qkv = (const uint4*)base; w.row_o = (const uint4*)(base + QKV);
            w.col_qkv = (const uint4*)(base + QKV + OW); w.col_o = (const uint4*)(base + 2 * QKV + OW);
            w.w1 = (const uint4*)(base + 2 * QKV + 2 * OW); w.w2 = (const uint4*)(base + 2 * QKV + 2 * OW + W1);
            w.row_qkvb = B0 + lo[l].a[0].qkvb; w.col_qkvb = B0 + lo[l].a[1].qkvb;
        }
    }
    *out = m;
    return NNJ_OK;
}

void nnj_model_destroy(nnj_model* m) {
    if (!m) return;
    DeviceGuard guard(m->device);
    if (m->blob) cudaFree(m->blob);
    if (m->blob_bf) cudaFree(m->blob_bf);
    if (m->blob_enc) cudaFree(m->blob_enc);
    if (m->host_ws) cudaFree(m->host_ws);
    for (cudaEvent_t e : m->host_events) cudaEventDestroy(e);
    if (m->host_compute) cudaStreamDestroy(m->host_compute);
    if (m->host_copy) cudaStreamDestroy(m->host_copy);
    delete m;
}

int64_t nnj_workspace_bytes(const nnj_model* m, int what, int B, int R, int L) {
    if (!m || B < 1 || R < 2 || L < 1) return set_error(NNJ_ERR_INVALID, "workspace_bytes: bad arguments");
    switch (what) {
        case 0: return (int64_t)encoder_ws_bytes(m, B, R, L);
        case 1: return (int64_t)nj_scores_ws_bytes(m, B, R, L, 0);
        case 2: return (int64_t)nj_rollout_ws_bytes(m, B, R, L);
        default: return set_error(NNJ_ERR_INVALID, "workspace_bytes: unknown selector");
    }
}

#define CHECK_ARGS(cond, msg) \
    do { if (!(cond)) return set_error(NNJ_ERR_INVALID, msg); } while (0)
// every compute entry point runs on the model's device whatever the caller's current device is
#define ON_MODEL_DEVICE(m)                                                              \
    DeviceGuard guard_((m)->device);                                                    \
    if (guard_.err != cudaSuccess) return set_cuda_error(guard_.err, __FILE__, __LINE__)

int nnj_encode(nnj_model* m, const int8_t* data, const uint8_t* mask, int B, int R, int L, float* out, void* ws, int64_t ws_bytes,
               void* stream) {
    CHECK_ARGS(m && data && out && ws && B >= 1 && R >= 2 && L >= 1, "encode: bad arguments");
    ON_MODEL_DEVICE(m);
    return run_encoder(m, data, mask, B, R, L, out, (size_t)R * L * D, ws, (size_t)ws_bytes, (cudaStream_t)stream);
}

int nnj_pair_scores_full(nnj_model* m, const float* state, const uint8_t* mask, int B, int Rp, int C, float* logits, void* ws,
                         int64_t ws_bytes, void* stream) {
    CHECK_ARGS(m && state && logits && ws && B >= 1, "pair_scores_full: bad arguments");
    ON_MODEL_DEVICE(m);
    return run_pair_scores(m, state, mask, B, Rp, C, nullptr, nullptr, 0, true, logits, ws, (size_t)ws_bytes, (cudaStream_t)stream);
}

int nnj_pair_scores_list(nnj_model* m, const float* state, const uint8_t* mask, int B, int Rp, int C, const int32_t* pi,
                         const int32_t* pj, int N, float* scores, void* ws, int64_t ws_bytes, void* stream) {
    CHECK_ARGS(m && state && scores && ws && pi && pj && B >= 1 && N >= 1, "pair_scores_list: bad arguments");
    ON_MODEL_DEVICE(m);
    return run_pair_scores(m, state, mask, B, Rp, C, pi, pj, N, false, scores, ws, (size_t)ws_bytes, (cudaStream_t)stream);
}

int nnj_pair_scores_incr(nnj_model* m, const float* state, const uint8_t* mask, int B, int Rp, int C, const int32_t* prev_ij,
                         const float* logits_prev, float* logits_out, void* ws, int64_t ws_bytes, void* stream) {
    CHECK_ARGS(m && state && prev_ij && logits_prev && logits_out && ws && B >= 1, "pair_scores_incr: bad arguments");
    ON_MODEL_DEVICE(m);
    return run_pair_scores_incr(m, state, mask, B, Rp, C, prev_ij, logits_prev, logits_out, ws, (size_t)ws_bytes, (cudaStream_t)stream);
}

int nnj_aggregate(nnj_model* m, const float* state, int B, int Rp, int C, const int32_t* ij, float* out, void* ws, int64_t ws_bytes,
                  void* stream) {
    CHECK_ARGS(m && state && ij && out && ws && B >= 1, "aggregate: bad arguments");
    ON_MODEL_DEVICE(m);
    return run_aggregate(m, state, B, Rp, C, ij, out, (size_t)C * D, ws, (size_t)ws_bytes, (cudaStream_t)stream);
}

int nnj_merge(nnj_model* m, const float* state_in, int B, int Rp, int C, const int32_t* ij, float* state_out, void* ws,
              int64_t ws_bytes, void* stream) {
    CHECK_ARGS(m && state_in && ij && state_out && ws && B >= 1 && Rp >= 3, "merge: bad arguments (need R' >= 3)");
    ON_MODEL_DEVICE(m);
    return run_merge(m, state_in, B, Rp, C, ij, state_out, ws, (size_t)ws_bytes, (cudaStream_t)stream);
}

int nnj_rollout(nnj_model* m, const int8_t* data, const uint8_t* mask, int B, int R, int L, int select_mode, const float* gumbel,
                int32_t* merges, float* logits_trace, float* selected_logp, void* ws, int64_t ws_bytes, void* stream) {
    CHECK_ARGS(m && data && merges && ws && B >= 1 && R >= 2 && L >= 1, "rollout: bad arguments");
    ON_MODEL_DEVICE(m);
    return run_rollout(m, data, nullptr, mask, B, R, L, select_mode, gumbel, merges, logits_trace, selected_logp, ws, (size_t)ws_bytes,
                       (cudaStream_t)stream);
}

int nnj_rollout_from_state(nnj_model* m, const float* state, const uint8_t* mask, int B, int R, int C, int select_mode,
                           const float* gumbel, int32_t* merges, float* logits_trace, float* selected_logp, void* ws,
                           int64_t ws_bytes, void* stream) {
    CHECK_ARGS(m && state && merges && ws && B >= 1 && R >= 2 && C >= 1, "rollout_from_state: bad arguments");
    ON_MODEL_DEVICE(m);
    return run_rollout(m, nullptr, state, mask, B, R, C, select_mode, gumbel, merges, logits_trace, selected_logp, ws, (size_t)ws_bytes,
                       (cudaStream_t)stream);
}

int nnj_gemm_split_bf16(const float* A, const float* B, float* Cm, int Z, int M, int N, int K, void* ws, int64_t ws_bytes, void* stream) {
    CHECK_ARGS(A && B && Cm && ws && Z >= 1 && M >= 1 && N >= 1 && K >= 8, "gemm_split_bf16: bad arguments");
    return run_gemm_split_bf16(A, B, Cm, Z, M, N, K, ws, (size_t)ws_bytes, (cudaStream_t)stream);
}

int64_t nnj_llh_workspace_bytes(int B, int R, int L) { return (B >= 1 && R >= 3 && L >= 1) ? (int64_t)llh_ws_bytes(B, R, L) : -1; }

int nnj_llh_eval(const uint8_t* tips, const double* weights, const int32_t* children_h, const double* brlen_h, const double* model_h, int B, int R, int L,
                 double* llh_h, void* ws, int64_t ws_bytes, void* stream) {
    CHECK_ARGS(tips && weights && children_h && brlen_h && model_h && llh_h && ws && B >= 1 && R >= 3 && R <= 4096 && L >= 1, "llh_eval: bad arguments");
    const LlhTrees in{tips, weights, children_h, const_cast<double*>(brlen_h), const_cast<double*>(model_h), B, R, L};
    return run_llh(in, LlhMode::Eval, {}, nullptr, llh_h, ws, (size_t)ws_bytes, (cudaStream_t)stream);
}

int nnj_llh_optimize_brlen(const uint8_t* tips, const double* weights, const int32_t* children_h, double* brlen_h, const double* model_h, int B, int R, int L,
                           int max_passes, double eps, double* llh_before_h, double* llh_after_h, void* ws, int64_t ws_bytes, void* stream) {
    CHECK_ARGS(tips && weights && children_h && brlen_h && model_h && llh_after_h && ws && B >= 1 && R >= 3 && R <= 4096 && L >= 1 && max_passes >= 1,
               "llh_optimize_brlen: bad arguments");
    const LlhTrees in{tips, weights, children_h, brlen_h, const_cast<double*>(model_h), B, R, L};
    return run_llh(in, LlhMode::Brlen, {max_passes, eps, 0.0, 0}, llh_before_h, llh_after_h, ws, (size_t)ws_bytes, (cudaStream_t)stream);
}

int nnj_llh_optimize_all(const uint8_t* tips, const double* weights, const int32_t* children_h, double* brlen_h, double* model_h, int B, int R, int L,
                         int max_passes, double eps, double lh_eps, int max_rounds, double* llh_before_h, double* llh_after_h, void* ws, int64_t ws_bytes,
                         void* stream) {
    CHECK_ARGS(tips && weights && children_h && brlen_h && model_h && llh_after_h && ws && B >= 1 && R >= 3 && R <= 4096 && L >= 1 && max_passes >= 1 && max_rounds >= 1,
               "llh_optimize_all: bad arguments");
    const LlhTrees in{tips, weights, children_h, brlen_h, model_h, B, R, L};
    return run_llh(in, LlhMode::All, {max_passes, eps, lh_eps, max_rounds}, llh_before_h, llh_after_h, ws, (size_t)ws_bytes, (cudaStream_t)stream);
}

int64_t nnj_llh_support_workspace_bytes(int B, int R, int L, int n_rell) {
    return (B >= 1 && R >= 3 && L >= 1 && n_rell >= 0) ? (int64_t)llh_support_ws_bytes(B, R, L, n_rell) : -1;
}

int nnj_llh_branch_support(const uint8_t* tips, const double* weights, const int32_t* children_h, const double* brlen_h, const double* model_h, int B, int R,
                           int L, uint64_t seed, int64_t rep0, int n_rell, int32_t* branch_node_h, double* llh_h, double* nni_brlen_h, int32_t* sh_count_h,
                           int32_t* lbp_count_h, double* site_llh_dev, void* ws, int64_t ws_bytes, void* stream) {
    CHECK_ARGS(tips && weights && children_h && brlen_h && model_h && ws && B >= 1 && R >= 3 && R <= 4096 && L >= 1 && n_rell >= 0 && rep0 >= 0 &&
               (R == 3 || (branch_node_h && llh_h && nni_brlen_h && sh_count_h && lbp_count_h)), "llh_branch_support: bad arguments");
    const LlhTrees in{tips, weights, children_h, const_cast<double*>(brlen_h), const_cast<double*>(model_h), B, R, L};
    return run_llh_support(in, seed, rep0, n_rell, branch_node_h, llh_h, nni_brlen_h, sh_count_h, lbp_count_h, site_llh_dev, ws, (size_t)ws_bytes,
                           (cudaStream_t)stream);
}

static bool topo_shape_ok(int K, int R, int L, int n_boot) { return K >= 2 && K <= 1024 && R >= 4 && R <= 4096 && L >= 1 && n_boot >= 1 && n_boot <= 1000000; }

int64_t nnj_llh_topotest_workspace_bytes(int K, int R, int L, int n_boot) {
    return topo_shape_ok(K, R, L, n_boot) ? (int64_t)llh_topo_ws_bytes(K, R, L, n_boot) : -1;
}

int nnj_llh_topology_test(const uint8_t* tips, const double* weights, const int32_t* children_h, const double* brlen_h, const double* model_h, int K, int R,
                          int L, uint64_t seed, int n_boot, double* llh_h, int32_t* win_h, int32_t* kh_h, int32_t* sh_h, double* elw_h, double* site_llh_dev,
                          void* ws, int64_t ws_bytes, void* stream) {
    CHECK_ARGS(tips && weights && children_h && brlen_h && model_h && llh_h && win_h && kh_h && sh_h && elw_h && ws && topo_shape_ok(K, R, L, n_boot),
               "llh_topology_test: bad arguments (2 <= K <= 1024, 4 <= R <= 4096, 1 <= n_boot <= 10^6)");
    return run_llh_topo(tips, weights, children_h, brlen_h, model_h, K, R, L, seed, n_boot, llh_h, win_h, kh_h, sh_h, elw_h, site_llh_dev, ws,
                        (size_t)ws_bytes, (cudaStream_t)stream);
}

int nnj_gamma_rates(double alpha, int ncat, double* rates_h) {
    CHECK_ARGS(rates_h, "gamma_rates: bad arguments");
    return gamma_rates(alpha, ncat, rates_h);
}

int64_t nnj_rank_loss_workspace_bytes(int B, int R) { return (B >= 1 && R >= 3 && R <= 256) ? (int64_t)rank_loss_ws_bytes(B, R) : -1; }

int nnj_rank_loss(const float* logits_trace, const uint8_t* in_set, int B, int R, float margin, double ratio, float* out, void* ws, int64_t ws_bytes,
                  void* stream) {
    CHECK_ARGS(logits_trace && in_set && out && ws && B >= 1, "rank_loss: bad arguments");
    return run_rank_loss(logits_trace, in_set, B, R, margin, ratio, out, ws, (size_t)ws_bytes, (cudaStream_t)stream);
}

int nnj_bootstrap_columns(const int8_t* data, int R, int L, int l_eff, uint64_t seed, int64_t rep0, int B, int8_t* out, void* stream) {
    CHECK_ARGS(data && out && R >= 1 && L >= 1 && l_eff >= 1 && l_eff <= L && B >= 1 && rep0 >= 0 && rep0 <= INT64_MAX - B &&
               ((uintptr_t)data & 3) == 0 && ((uintptr_t)out & 3) == 0, "bootstrap_columns: bad arguments");
    return run_bootstrap_columns(data, R, L, l_eff, seed, rep0, B, out, (cudaStream_t)stream);
}

int nnj_split_distances(const int32_t* merges, int B, int R, const uint64_t* splits, int S, int32_t* dist, void* stream) {
    CHECK_ARGS(merges && B >= 1 && S >= 0 && (S == 0 || (splits && dist)), "split_distances: bad arguments");
    return run_split_distances(merges, B, R, splits, S, dist, (cudaStream_t)stream);
}

int nnj_tc_selftest(const float* A, const float* B, float* Dm, int N, void* stream) {
    CHECK_ARGS(A && B && Dm, "tc_selftest: bad arguments");
    return run_tc_unit(A, B, Dm, N, (cudaStream_t)stream);
}

int nnj_rollout_host(nnj_model* m, const int8_t* data_h, const uint8_t* mask_h, int B, int R, int L, int select_mode,
                     const float* gumbel_h, int32_t* merges_h, float* selected_logp_h) {
    CHECK_ARGS(m && data_h && merges_h && B >= 1 && R >= 2 && L >= 1, "rollout_host: bad arguments");
    ON_MODEL_DEVICE(m);
    std::lock_guard<std::mutex> lock(m->host_lock);          // the workspace and the streams below belong to the model
    // The batch is processed in the library's rollout chunks.  Chunk i+1 is staged host -> device on a copy stream while chunk i
    // runs on a compute stream (both non-blocking: the caller's streams, PyTorch's included, are not serialised against).
    const int chunk = nj_rollout_chunk(m, B, R, L);
    const int n_chunks = (B + chunk - 1) / chunk;
    const size_t ws_bytes = nj_rollout_ws_bytes(m, chunk, R, L);
    const size_t P0 = (size_t)R * (R - 1) / 2;
    const size_t t_data = (size_t)R * L * 4, t_mask = (size_t)L, t_mg = (size_t)(R - 1) * 2, t_gum = gumbel_h ? (size_t)(R - 1) * P0 : 0;
    // workspace + staging buffers live in one grow-only allocation owned by the model (no cudaMalloc on the steady-state path)
    auto staging = [&](char* base) {
        WsCarver c(base);
        c.take<char>(ws_bytes);                                   // the rollout workspace
        struct { int8_t* data; uint8_t* mask; int32_t* mg; float *slp, *gum; size_t end; } io;
        io.data = c.take<int8_t>(B * t_data);
        io.mask = c.take<uint8_t>(B * t_mask);
        io.mg = c.take<int32_t>(B * t_mg);
        io.slp = c.take<float>((size_t)B * (R - 1));
        io.gum = c.take<float>(B * t_gum);
        io.end = c.off + 256;
        return io;
    };
    const size_t need = staging(nullptr).end;
    if (m->host_ws_bytes < need) {
        if (m->host_ws) { CUDA_TRY(cudaDeviceSynchronize()); cudaFree(m->host_ws); m->host_ws = nullptr; m->host_ws_bytes = 0; }
        CUDA_TRY(cudaMalloc(&m->host_ws, need));
        m->host_ws_bytes = need;
    }
    if (!m->host_compute) CUDA_TRY(cudaStreamCreateWithFlags(&m->host_compute, cudaStreamNonBlocking));
    if (!m->host_copy) CUDA_TRY(cudaStreamCreateWithFlags(&m->host_copy, cudaStreamNonBlocking));
    while ((int)m->host_events.size() < n_chunks) {
        cudaEvent_t ev;
        CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        m->host_events.push_back(ev);
    }
    char* ws = reinterpret_cast<char*>(m->host_ws);
    const auto io = staging(ws);
    int8_t* d_data = io.data;
    uint8_t* d_mask = io.mask;
    int32_t* d_mg = io.mg;
    float* d_slp = io.slp;
    float* d_gum = gumbel_h ? io.gum : nullptr;
    cudaStream_t cs = m->host_compute, xs = m->host_copy;
    cudaError_t e = cudaSuccess;
    int rc = NNJ_OK;
    do {
        for (int c = 0; c < n_chunks && e == cudaSuccess; ++c) {      // all H2D copies are queued up front, one event per chunk
            const size_t b0 = (size_t)c * chunk, nb = (size_t)((B - (int)b0 < chunk) ? (B - (int)b0) : chunk);
            if ((e = cudaMemcpyAsync(d_data + b0 * t_data, data_h + b0 * t_data, nb * t_data, cudaMemcpyHostToDevice, xs)) != cudaSuccess) break;
            if (mask_h && (e = cudaMemcpyAsync(d_mask + b0 * t_mask, mask_h + b0 * t_mask, nb * t_mask, cudaMemcpyHostToDevice, xs)) != cudaSuccess) break;
            if (gumbel_h && (e = cudaMemcpyAsync(d_gum + b0 * t_gum, gumbel_h + b0 * t_gum, nb * t_gum * 4, cudaMemcpyHostToDevice, xs)) != cudaSuccess) break;
            if (select_mode == NNJ_SELECT_FORCED &&      // teacher forcing: the merge lists are inputs as well
                (e = cudaMemcpyAsync(d_mg + b0 * t_mg, merges_h + b0 * t_mg, nb * t_mg * 4, cudaMemcpyHostToDevice, xs)) != cudaSuccess) break;
            e = cudaEventRecord(m->host_events[c], xs);
        }
        if (e != cudaSuccess) break;
        for (int c = 0; c < n_chunks; ++c) {
            const size_t b0 = (size_t)c * chunk;
            const int nb = (B - (int)b0 < chunk) ? (B - (int)b0) : chunk;
            if ((e = cudaStreamWaitEvent(cs, m->host_events[c], 0)) != cudaSuccess) break;
            rc = run_rollout(m, d_data + b0 * t_data, nullptr, mask_h ? d_mask + b0 * t_mask : nullptr, nb, R, L, select_mode,
                             d_gum ? d_gum + b0 * t_gum : nullptr, d_mg + b0 * t_mg, nullptr, selected_logp_h ? d_slp + b0 * (R - 1) : nullptr,
                             ws, ws_bytes, cs);
            if (rc != NNJ_OK) break;
            // results of this chunk go home while the next chunk computes
            if ((e = cudaMemcpyAsync(merges_h + b0 * t_mg, d_mg + b0 * t_mg, (size_t)nb * t_mg * 4, cudaMemcpyDeviceToHost, cs)) != cudaSuccess) break;
            if (selected_logp_h && (e = cudaMemcpyAsync(selected_logp_h + b0 * (R - 1), d_slp + b0 * (R - 1), (size_t)nb * (R - 1) * 4,
                                                        cudaMemcpyDeviceToHost, cs)) != cudaSuccess) break;
        }
        if (rc != NNJ_OK || e != cudaSuccess) break;
        e = cudaStreamSynchronize(cs);
    } while (0);
    if (rc != NNJ_OK || e != cudaSuccess) { cudaStreamSynchronize(xs); cudaStreamSynchronize(cs); }
    if (rc != NNJ_OK) return rc;
    if (e != cudaSuccess) return set_cuda_error(e, __FILE__, __LINE__);
    return NNJ_OK;
}

}  // extern "C"
