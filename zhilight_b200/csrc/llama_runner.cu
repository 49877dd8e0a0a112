// Host-side decode driver (C++): weights, KV buffers, the per-step kernel chain and its CUDA graph.
//
// Stands in for model::LLaMA::encode / EncoderLayer::forward / Attention::dynamic_batch_forward /
// FeedForward::forward at decode (reference src/model/llama.cpp:75-165, src/nn/block/block.cpp:86-143,
// src/nn/attention/attention.cpp:846-964, src/nn/feedforward/feedforward.cpp:113-137) and for the
// Int4GPTQ load pipeline (src/nn/linear/linear.cpp:1139-1244).  The reference launches ~12 kernels per
// layer with no graph; here a layer is 8 launches chained with programmatic dependent launch inside one
// CUDA graph per batch size.
#include "common.cuh"
#include "w4_layout.cuh"
#include "comm_dev.cuh"

#include <cstdlib>
#include <cstring>
#include <map>
#include <utility>
#include <string>
#include <vector>

extern unsigned long long* g_w4_trace;   // debug timeline buffer (zl_w4_set_trace)

namespace {

struct Staged {
    void* ptr = nullptr;
    int rows = 0, cols = 0, elem = 0;
};

struct W4Lin {
    void* packed = nullptr;     // ZLW4  (fp16 HMMA kernels) -- only kept when some batch size needs it
    void* packed_i = nullptr;   // ZLW4I (exact-integer IMMA kernel, small M)
    void* bias = nullptr;
    int N = 0, K = 0;
};
struct DenseLin {
    void* w = nullptr;
    void* bias = nullptr;
    int N = 0, K = 0;
    // W8A8 (quant_type 2 / 7): 8-bit weights (N, K) + per-row scales; w is released
    void* w8 = nullptr;
    void* w_scale = nullptr;   // int8: (N) in the activation dtype (linear.cpp:541); fp8: (N) f32 rows
    int w8_kind = -1;          // ZL_W8_INT8 or ZL_W8_FP8_ROWS
};

struct Layer {
    void* ln_attn = nullptr;
    void* ln_ff = nullptr;
    W4Lin q_qkv, q_o, q_gu, q_down;
    DenseLin d_qkv, d_o, d_gu, d_down;
    void* kbuf = nullptr;   // (max_batch, max_seq, Hkv, d)
    void* vbuf = nullptr;
    void** k_addrs = nullptr;   // device (max_batch)
    void** v_addrs = nullptr;
};

}  // namespace

struct zl_llama {
    zl_llama_config_t cfg{};
    cudaStream_t stream = nullptr;
    std::map<std::string, Staged> staged;
    std::vector<Layer> layers;
    void* emb = nullptr;
    void* lm_head = nullptr;
    void* ln_f = nullptr;
    bool lm_head_tied = false;
    bool finalized = false;
    // local (per-rank) sizes
    int hq = 0, hkv = 0, ff = 0;
    // activations
    void* h2 = nullptr;   // second residual-stream buffer: the fused TP exchange ping-pongs between h and h2
    void *h = nullptr, *xn = nullptr, *qkv = nullptr, *q = nullptr, *ao = nullptr, *act = nullptr,
         *pend = nullptr, *gu = nullptr;
    float* logits = nullptr;
    float *cosb = nullptr, *sinb = nullptr;
    int32_t *d_tokens = nullptr, *d_pos = nullptr, *d_lens = nullptr, *d_next = nullptr, *d_iota = nullptr;
    void* attn_ws = nullptr;
    size_t attn_ws_bytes = 0;
    void* argmax_ws = nullptr;
    int32_t* h_stage = nullptr;   // pinned: tokens | pos | lens | next
    // zl_llama_set_state staging: pinned H2D copies read the host buffer when they EXECUTE, so a set_state -> step_device
    // loop that runs ahead of the GPU must not rewrite a slot whose copy is still queued: ring of slots, one event each
    static constexpr int kStageSlots = 8;
    int32_t* h_ring = nullptr;    // pinned [kStageSlots][2 * max_batch]
    cudaEvent_t ring_ev[kStageSlots] = {};
    bool ring_used[kStageSlots] = {};
    int ring_next = 0;
    // prefill keeps its own (token, position) arrays: the decode-state arrays d_tokens / d_pos of tasks 0..B-1 survive a
    // prefill that happens between two zl_llama_step_device calls (continuous batching)
    int32_t *d_pf_tokens = nullptr, *d_pf_pos = nullptr;
    const int32_t* cur_pos = nullptr;      // positions of the launch sequence being enqueued (d_pos or d_pf_pos)
    const int32_t* cur_tokens = nullptr;
    zl_comm_t* comm = nullptr;            // TP exchange (set by zl_llama_set_comm when tp_size > 1)
    int vshard = 0;                       // vocabulary rows of lm_head held by this rank
    void* cand = nullptr;                 // [B] {float value, int index} local argmax candidates
    void* cand_all = nullptr;             // [tp][B] gathered candidates
    std::map<long long, cudaGraphExec_t> graphs;   // key = B * 2^33 + sampling * 2^32 + attention length bucket
    int cur_max_len = 0;                            // host-side upper bound of buf_lens (positions + 1)
    double weight_bytes = 0;
    int kernels_per_step = 0;
    // chunked prefill (cfg.prefill_chunk > 0): activation buffers hold tok_cap = max(max_batch, chunk) tokens
    int tok_cap = 0;
    // dual-stream chunked prefill (EncoderLayer::dual_stream_encode, block.cpp:205-441): compute stream = m->stream
    cudaStream_t reduce_stream = nullptr;
    cudaEvent_t ev_o[2] = {nullptr, nullptr}, ev_r1[2] = {nullptr, nullptr}, ev_dn[2] = {nullptr, nullptr},
                ev_r2[2] = {nullptr, nullptr};
    void* xq = nullptr;           // W8A8: quantised activations of the Linear being run (tok_cap x max K bytes)
    float* xs = nullptr;          //       their scales (tok_cap)
    int32_t* d_tb = nullptr;      // token -> task map of the chunk being prefilled
    const int32_t* cur_tb = nullptr;   // token -> task map of the launch sequence being enqueued (d_iota at decode)
    int8_t* d_mask = nullptr;     // (chunk, max_seq) causal mask of the chunk
    // sampling (zl_llama_set_sampling): per-task parameters, seen-token bits and draw counters on the device, read by
    // the graph at replay time; a host flag per task selects the zl_sample graph for batches that hold such a task
    zl_sample_params_t* d_sparams = nullptr;   // (max_batch)
    uint32_t* d_seen = nullptr;                // (max_batch, ceil(vshard / 32))
    uint32_t* d_draws = nullptr;               // (max_batch)
    std::vector<char> sampling;                // (max_batch) task has non-default sampling state
};

namespace {

using namespace zl;

#define RCHECK(expr)                \
    do {                            \
        int _rc = (expr);           \
        if (_rc != ZL_OK) return _rc; \
    } while (0)



int dmalloc(void** p, size_t bytes) {
    ZL_CHECK_CUDA(cudaMalloc(p, bytes ? bytes : 16));
    return ZL_OK;
}

__global__ void k_lens_from_pos(const int32_t* __restrict__ pos, int32_t* __restrict__ lens, int B,
                                unsigned long long* trace) {
    pdl_trigger();
    pdl_wait();
    if (trace && blockIdx.x == 0 && threadIdx.x == 0) trace[1] = globaltimer_ns();   // debug timeline: step start
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < B) lens[i] = pos[i] + 1;
}
__global__ void k_advance(int32_t* __restrict__ tokens, int32_t* __restrict__ pos, const int32_t* __restrict__ next,
                          int B, unsigned long long* trace) {
    if (trace && blockIdx.x == 0 && threadIdx.x == 0 && trace[2] == 0) trace[2] = globaltimer_ns();   // debug: first step end
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < B) {
        tokens[i] = next[i];
        pos[i] += 1;
    }
}
// prefill chunk setup: positions pos0.., token -> task map, the task's buffer length, and the causal mask
// mask[i][j] = j <= pos0 + i over len_buf = pos0 + n keys (attention_kernel.cu:434-489 mask contract, int8)
__global__ void k_prefill_setup(int32_t* __restrict__ pos, int32_t* __restrict__ tb, int32_t* __restrict__ lens,
                                int8_t* __restrict__ mask, int task, int pos0, int n) {
    const int len_buf = pos0 + n;
    for (int i = threadIdx.x + blockIdx.x * blockDim.x; i < n * len_buf; i += blockDim.x * gridDim.x) {
        const int qi = i / len_buf, j = i % len_buf;
        mask[i] = j <= pos0 + qi ? 1 : 0;
    }
    if (blockIdx.x == 0) {
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            pos[i] = pos0 + i;
            tb[i] = task;
        }
        if (threadIdx.x == 0) lens[task] = len_buf;
    }
}

template <typename T>
__global__ void k_f32_to_t(const float* __restrict__ in, T* __restrict__ out, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = from_f32<T>(in[i]);
}
__global__ void k_fill_from_scalar(float* __restrict__ dst, int n, const float* __restrict__ scalar) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = *scalar;
}
__global__ void k_and_u32(uint32_t* __restrict__ p, size_t n, uint32_t mask) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] &= mask;
}
__global__ void k_set_f32(float* p, float v) { *p = v; }
// synthetic symmetric checkpoints: a uniformly random nibble minus the fixed zero point 8 has mean -0.5, and with thousands
// of such weights per row every layer adds a common-mode offset to the residual stream that overflows fp16 after ~30
// layers (measured: NaN logits on the 32-layer model).  Nibble 0 -> 8 makes q - 8 symmetric around zero (-7 .. 7).
__global__ void k_recentre_nibbles(uint32_t* __restrict__ p, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const uint32_t w = p[i];
        const uint32_t zero = ~(w | (w >> 1) | (w >> 2) | (w >> 3)) & 0x11111111u;
        p[i] = w | (zero << 3);
    }
}

__global__ void k_iota(int32_t* p, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = i;
}
__global__ void k_ptr_table(void** tab, char* base, size_t stride, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) tab[i] = base + (size_t)i * stride;
}
__global__ void k_swiglu_row_map(int32_t* map, int F) {
    // packed row p: 16-row tile = 8 gate rows then the 8 matching up rows (source = [gate(F); up(F)])
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < 2 * F) {
        int tile = p >> 4, r = p & 15;
        map[p] = (r < 8) ? tile * 8 + r : F + tile * 8 + (r - 8);
    }
}

const Staged* find(const zl_llama* m, const std::string& name) {
    auto it = m->staged.find(name);
    return it == m->staged.end() ? nullptr : &it->second;
}

void drop(zl_llama* m, const std::string& name) {
    auto it = m->staged.find(name);
    if (it != m->staged.end()) {
        cudaFree(it->second.ptr);
        m->staged.erase(it);
    }
}

// frees device temporaries on every exit path of a load helper
struct DevTmp {
    std::vector<void*> ptrs;
    ~DevTmp() {
        for (void* p : ptrs)
            if (p) cudaFree(p);
    }
    int alloc(void** p, size_t bytes) {
        int rc = dmalloc(p, bytes);
        if (rc == ZL_OK) ptrs.push_back(*p);
        return rc;
    }
};

int fail_state(int line, const std::string& msg, int code = ZL_ERR_STATE) {
    zl_set_last_error(__FILE__, line, msg.c_str());
    return code;
}

// g_idx of a desc_act / act-order checkpoint is not k / group_size; the reference then gathers rows by argsort(g_idx)
// and permutes the activations at run time (linear.cpp:1092-1094, 1145-1146, 1168-1210).  The fused kernels here have no
// run-time activation permute, so such a checkpoint is rejected at load instead of producing garbage.
int check_g_idx_sequential(zl_llama* m, const std::string& prefix, int K) {
    const Staged* gi = find(m, prefix + ".g_idx");
    if (!gi) return ZL_OK;
    if ((size_t)gi->rows * gi->cols != (size_t)K || gi->elem != 4)
        return fail_state(__LINE__, "ill-shaped g_idx for " + prefix + " (expected K int32)");
    std::vector<int32_t> host(K);
    ZL_CHECK_CUDA(cudaMemcpyAsync(host.data(), gi->ptr, (size_t)K * 4, cudaMemcpyDeviceToHost, m->stream));
    ZL_CHECK_CUDA(cudaStreamSynchronize(m->stream));
    for (int k = 0; k < K; ++k)
        if (host[k] != k / m->cfg.group_size)
            return fail_state(__LINE__, "act-order (desc_act) GPTQ checkpoint: " + prefix +
                                            ".g_idx is not sequential; not supported by the fused W4 kernels",
                              ZL_ERR_UNSUPPORTED);
    return ZL_OK;
}

// HF GPTQ/AWQ tensors of one Linear -> reference k-major tensors written at row offset n_off of the fused
// k-major buffers (linear.cpp:1139-1160 preprocess_weight + 1085-1099 transpose_weight).
int to_k_major(zl_llama* m, const std::string& prefix, int K, int N, uint32_t* qw_km, uint8_t* qz_km, __half* sc_km,
               int n_off, int n_total) {
    const Staged* qw = find(m, prefix + ".qweight");
    const Staged* qz = find(m, prefix + ".qzeros");
    const Staged* sc = find(m, prefix + ".scales");
    if (!qw || !qz || !sc) return fail_state(__LINE__, "missing GPTQ tensors for " + prefix);
    const int G = K / m->cfg.group_size;
    const bool awq = m->cfg.quant_type == 6;
    // every shape / element size is validated BEFORE the first kernel touches the tensors (in-place transforms below)
    const bool qw_ok = awq ? (qw->rows == K && qw->cols == N / 8) : (qw->rows == K / 8 && qw->cols == N);
    if (!qw_ok || qw->elem != 4) return fail_state(__LINE__, "ill-shaped qweight for " + prefix, ZL_ERR_INVALID_ARG);
    if (qz->rows != G || qz->cols != N / 8 || qz->elem != 4)
        return fail_state(__LINE__, "ill-shaped qzeros for " + prefix + " (expected (K/g, N/8) int32)", ZL_ERR_INVALID_ARG);
    if (sc->rows != G || sc->cols != N || sc->elem != 2)
        return fail_state(__LINE__, "ill-shaped scales for " + prefix + " (expected (K/g, N) fp16)", ZL_ERR_INVALID_ARG);
    RCHECK(check_g_idx_sequential(m, prefix, K));
    cudaStream_t st = m->stream;
    DevTmp tmp;
    uint32_t* w_kn = nullptr;   // (K/8, N)
    if (awq) {
        RCHECK(tmp.alloc((void**)&w_kn, (size_t)(K / 8) * N * 4));
        RCHECK(zl_awq_shuffle((const uint32_t*)qw->ptr, w_kn, K, N, 1, st));
        RCHECK(zl_awq_un_shuffle((uint32_t*)qz->ptr, G, N / 8, st));
    } else {
        w_kn = (uint32_t*)qw->ptr;
        RCHECK(zl_gptq_shuffle(w_kn, nullptr, nullptr, K, N, st));
        RCHECK(zl_gptq_increase_zero((uint32_t*)qz->ptr, (size_t)G * (N / 8), st));
    }
    uint8_t* z8 = nullptr;   // (G, N)
    RCHECK(tmp.alloc((void**)&z8, (size_t)G * N));
    RCHECK(zl_q4_to_q8((const uint32_t*)qz->ptr, z8, (size_t)G * (N / 8), st));
    // transposes straight into the fused buffers (row offset n_off)
    RCHECK(zl_transpose_2d(w_kn, qw_km + (size_t)n_off * (K / 8), K / 8, N, 4, st));
    RCHECK(zl_transpose_2d(z8, qz_km + (size_t)n_off * G, G, N, 1, st));
    RCHECK(zl_transpose_2d(sc->ptr, sc_km + (size_t)n_off * G, G, N, 2, st));
    ZL_CHECK_CUDA(cudaStreamSynchronize(st));
    (void)n_total;
    return ZL_OK;
}

int build_w4(zl_llama* m, const std::vector<std::string>& prefixes, const std::vector<int>& ns, int K, bool swiglu,
             W4Lin* out, bool qkv_rope = false) {
    int N = 0;
    for (int n : ns) N += n;
    const int G = K / m->cfg.group_size;
    uint32_t* qw_km = nullptr;
    uint8_t* qz_km = nullptr;
    __half* sc_km = nullptr;
    DevTmp tmp;   // released on every exit path
    RCHECK(tmp.alloc((void**)&qw_km, (size_t)N * (K / 8) * 4));
    RCHECK(tmp.alloc((void**)&qz_km, (size_t)N * G));
    RCHECK(tmp.alloc((void**)&sc_km, (size_t)N * G * 2));
    int off = 0;
    bool any_bias = false;
    for (size_t i = 0; i < prefixes.size(); ++i) {
        RCHECK(to_k_major(m, prefixes[i], K, ns[i], qw_km, qz_km, sc_km, off, N));
        if (find(m, prefixes[i] + ".bias")) any_bias = true;
        off += ns[i];
    }
    int32_t* row_map = nullptr;
    if (swiglu) {
        RCHECK(tmp.alloc((void**)&row_map, (size_t)N * 4));
        k_swiglu_row_map<<<cdiv(N, 256), 256, 0, m->stream>>>(row_map, N / 2);
        ZL_CHECK_LAUNCH();
    } else if (qkv_rope) {
        RCHECK(tmp.alloc((void**)&row_map, (size_t)N * 4));
        RCHECK(zl_qkv_rope_row_map(row_map, N / m->cfg.dim_head, m->cfg.dim_head, m->stream));
    }
    const size_t pbytes = zl_w4_packed_bytes(N, K, m->cfg.group_size);
    ZL_CHECK_SUPPORTED(pbytes > 0);
    // the ZLW4I layout serves the exact-integer kernel (M <= 16 when its staged activations fit) and the tcgen05 kernel
    // (any M, N % 128 == 0); the fp16 mma.sync layout is only materialised when some launch size has neither
    const int m_max = m->cfg.prefill_chunk > m->cfg.max_batch ? m->cfg.prefill_chunk : m->cfg.max_batch;
    bool need_half = getenv("ZL_W4_FORCE_HALF") != nullptr;
    for (int mm = 1; mm <= (m_max < 17 ? m_max : 17); ++mm)
        if (!zl_w4_int_layout_route(mm, N, K)) need_half = true;
    RCHECK(dmalloc(&out->packed_i, pbytes));
    RCHECK(zl_w4_pack_v(qw_km, qz_km, sc_km, row_map, out->packed_i, N, K, m->cfg.group_size, m->cfg.sym, 1,
                        m->stream));
    if (need_half) {
        RCHECK(dmalloc(&out->packed, pbytes));
        RCHECK(zl_w4_pack_v(qw_km, qz_km, sc_km, row_map, out->packed, N, K, m->cfg.group_size, m->cfg.sym, 0,
                            m->stream));
    }
    if (any_bias && !swiglu) {
        RCHECK(dmalloc(&out->bias, (size_t)N * 2));
        ZL_CHECK_CUDA(cudaMemsetAsync(out->bias, 0, (size_t)N * 2, m->stream));
        off = 0;
        for (size_t i = 0; i < prefixes.size(); ++i) {
            const Staged* b = find(m, prefixes[i] + ".bias");
            if (b) {
                if ((size_t)b->rows * b->cols != (size_t)ns[i] || b->elem != 2)
                    return fail_state(__LINE__, "ill-shaped bias for " + prefixes[i], ZL_ERR_INVALID_ARG);
                ZL_CHECK_CUDA(cudaMemcpyAsync((char*)out->bias + (size_t)off * 2, b->ptr, (size_t)ns[i] * 2,
                                              cudaMemcpyDeviceToDevice, m->stream));
            }
            off += ns[i];
        }
        if (row_map) {   // the fused epilogues index bias by packed row
            void* pb = nullptr;
            RCHECK(dmalloc(&pb, (size_t)N * 2));
            RCHECK(zl_gather_rows_16(out->bias, row_map, pb, N, m->stream));
            ZL_CHECK_CUDA(cudaStreamSynchronize(m->stream));
            cudaFree(out->bias);
            out->bias = pb;
        }
    }
    ZL_CHECK_CUDA(cudaStreamSynchronize(m->stream));
    for (auto& p : prefixes) {
        drop(m, p + ".qweight");
        drop(m, p + ".qzeros");
        drop(m, p + ".scales");
        drop(m, p + ".g_idx");
        drop(m, p + ".bias");
    }
    out->N = N;
    out->K = K;
    m->weight_bytes += (double)pbytes;
    return ZL_OK;
}

int build_dense(zl_llama* m, const std::vector<std::string>& prefixes, const std::vector<int>& ns, int K,
                DenseLin* out) {
    int N = 0;
    for (int n : ns) N += n;
    RCHECK(dmalloc(&out->w, (size_t)N * K * 2));
    int off = 0;
    bool any_bias = false;
    for (size_t i = 0; i < prefixes.size(); ++i) {
        const Staged* w = find(m, prefixes[i] + ".weight");
        if (!w || w->rows != ns[i] || w->cols != K || w->elem != 2) {
            zl_set_last_error(__FILE__, __LINE__, ("missing/ill-shaped dense weight " + prefixes[i]).c_str());
            return ZL_ERR_STATE;
        }
        ZL_CHECK_CUDA(cudaMemcpyAsync((char*)out->w + (size_t)off * K * 2, w->ptr, (size_t)ns[i] * K * 2,
                                      cudaMemcpyDeviceToDevice, m->stream));
        if (find(m, prefixes[i] + ".bias")) any_bias = true;
        off += ns[i];
    }
    if (any_bias) {
        RCHECK(dmalloc(&out->bias, (size_t)N * 2));
        ZL_CHECK_CUDA(cudaMemsetAsync(out->bias, 0, (size_t)N * 2, m->stream));
        off = 0;
        for (size_t i = 0; i < prefixes.size(); ++i) {
            const Staged* b = find(m, prefixes[i] + ".bias");
            if (b)
                ZL_CHECK_CUDA(cudaMemcpyAsync((char*)out->bias + (size_t)off * 2, b->ptr, (size_t)ns[i] * 2,
                                              cudaMemcpyDeviceToDevice, m->stream));
            off += ns[i];
        }
    }
    ZL_CHECK_CUDA(cudaStreamSynchronize(m->stream));
    for (auto& p : prefixes) {
        drop(m, p + ".weight");
        drop(m, p + ".bias");
    }
    out->N = N;
    out->K = K;
    m->weight_bytes += (double)N * K * 2;
    return ZL_OK;
}

// quant_type 2 (AutoInt8, linear.cpp:521-550): the fp weight is quantised per output row at load with the same kernel
// as the activations; the scale is kept in the activation dtype (functions::typecast, linear.cpp:541).
int dense_to_int8(zl_llama* m, DenseLin* d) {
    const auto& c = m->cfg;
    float* sf = nullptr;
    RCHECK(dmalloc(&d->w8, (size_t)d->N * d->K));
    RCHECK(dmalloc((void**)&sf, (size_t)d->N * 4));
    RCHECK(dmalloc(&d->w_scale, (size_t)d->N * 2));
    RCHECK(zl_int8_quant_per_token(d->w, d->K, d->w8, sf, d->N, d->K, c.dtype, 0, m->stream));
    if (c.dtype == ZL_F16)
        k_f32_to_t<__half><<<cdiv(d->N, 256), 256, 0, m->stream>>>(sf, static_cast<__half*>(d->w_scale), d->N);
    else
        k_f32_to_t<__nv_bfloat16><<<cdiv(d->N, 256), 256, 0, m->stream>>>(sf, static_cast<__nv_bfloat16*>(d->w_scale), d->N);
    ZL_CHECK_LAUNCH();
    ZL_CHECK_CUDA(cudaStreamSynchronize(m->stream));
    cudaFree(sf);
    cudaFree(d->w);
    d->w = nullptr;
    d->w8_kind = ZL_W8_INT8;
    m->weight_bytes += (double)d->N * d->K + (double)d->N * 2 - (double)d->N * d->K * 2;
    return ZL_OK;
}

// quant_type 7 (Fp8Linear, linear.cpp:1612-1695): e4m3 weights + one f32 weight_scale per Linear.  Projections that
// share an input are fused along N with their scalar scales expanded to one scale per output row.
int build_fp8(zl_llama* m, const std::vector<std::string>& prefixes, const std::vector<int>& ns, int K, DenseLin* out) {
    int N = 0;
    for (int n : ns) N += n;
    RCHECK(dmalloc(&out->w8, (size_t)N * K));
    RCHECK(dmalloc(&out->w_scale, (size_t)N * 4));
    int off = 0;
    bool any_bias = false;
    for (size_t i = 0; i < prefixes.size(); ++i) {
        const Staged* w = find(m, prefixes[i] + ".weight");
        const Staged* ws = find(m, prefixes[i] + ".weight_scale");
        if (!w || w->rows != ns[i] || w->cols != K || w->elem != 1 || !ws || ws->elem != 4) {
            zl_set_last_error(__FILE__, __LINE__, ("missing/ill-shaped fp8 weight or weight_scale " + prefixes[i]).c_str());
            return ZL_ERR_STATE;
        }
        ZL_CHECK_CUDA(cudaMemcpyAsync((char*)out->w8 + (size_t)off * K, w->ptr, (size_t)ns[i] * K, cudaMemcpyDeviceToDevice,
                                      m->stream));
        k_fill_from_scalar<<<cdiv(ns[i], 256), 256, 0, m->stream>>>(static_cast<float*>(out->w_scale) + off, ns[i],
                                                                     static_cast<const float*>(ws->ptr));
        ZL_CHECK_LAUNCH();
        if (find(m, prefixes[i] + ".bias")) any_bias = true;
        off += ns[i];
    }
    if (any_bias) {
        RCHECK(dmalloc(&out->bias, (size_t)N * 2));
        ZL_CHECK_CUDA(cudaMemsetAsync(out->bias, 0, (size_t)N * 2, m->stream));
        off = 0;
        for (size_t i = 0; i < prefixes.size(); ++i) {
            const Staged* b = find(m, prefixes[i] + ".bias");
            if (b)
                ZL_CHECK_CUDA(cudaMemcpyAsync((char*)out->bias + (size_t)off * 2, b->ptr, (size_t)ns[i] * 2,
                                              cudaMemcpyDeviceToDevice, m->stream));
            off += ns[i];
        }
    }
    ZL_CHECK_CUDA(cudaStreamSynchronize(m->stream));
    for (auto& p : prefixes) {
        drop(m, p + ".weight");
        drop(m, p + ".weight_scale");
        drop(m, p + ".bias");
    }
    out->N = N;
    out->K = K;
    out->w8_kind = ZL_W8_FP8_ROWS;
    m->weight_bytes += (double)N * K + (double)N * 4;
    return ZL_OK;
}

int take_vector(zl_llama* m, const std::string& name, int n, void** out) {
    auto it = m->staged.find(name);
    if (it == m->staged.end() || (size_t)it->second.rows * it->second.cols != (size_t)n || it->second.elem != 2) {
        zl_set_last_error(__FILE__, __LINE__, ("missing/ill-shaped tensor " + name).c_str());
        return ZL_ERR_STATE;
    }
    *out = it->second.ptr;
    m->staged.erase(it);
    m->weight_bytes += (double)n * 2;
    return ZL_OK;
}

int finalize_layer(zl_llama* m, int l) {
    const auto& c = m->cfg;
    Layer& L = m->layers[l];
    const std::string p = "layers." + std::to_string(l) + ".";
    const int D = c.dim_model, d = c.dim_head;
    RCHECK(take_vector(m, p + "ln_attn.weight", D, &L.ln_attn));
    RCHECK(take_vector(m, p + "ln_ff.weight", D, &L.ln_ff));
    const std::vector<std::string> qkv = {p + "attn.project_q", p + "attn.project_k", p + "attn.project_v"};
    const std::vector<int> qkv_n = {m->hq * d, m->hkv * d, m->hkv * d};
    const std::vector<std::string> gu = {p + "ff.w_in", p + "ff.w_gated"};
    const std::vector<int> gu_n = {m->ff, m->ff};
    if (c.quant_type == 5 || c.quant_type == 6) {
        RCHECK(build_w4(m, qkv, qkv_n, D, false, &L.q_qkv, c.fuse >= 2));
        RCHECK(build_w4(m, {p + "attn.attn_out"}, {D}, m->hq * d, false, &L.q_o));
        RCHECK(build_w4(m, gu, gu_n, D, true, &L.q_gu));
        RCHECK(build_w4(m, {p + "ff.w_out"}, {D}, m->ff, false, &L.q_down));
    } else if (c.quant_type == 7) {
        RCHECK(build_fp8(m, qkv, qkv_n, D, &L.d_qkv));
        RCHECK(build_fp8(m, {p + "attn.attn_out"}, {D}, m->hq * d, &L.d_o));
        RCHECK(build_fp8(m, gu, gu_n, D, &L.d_gu));
        RCHECK(build_fp8(m, {p + "ff.w_out"}, {D}, m->ff, &L.d_down));
    } else {
        RCHECK(build_dense(m, qkv, qkv_n, D, &L.d_qkv));
        RCHECK(build_dense(m, {p + "attn.attn_out"}, {D}, m->hq * d, &L.d_o));
        RCHECK(build_dense(m, gu, gu_n, D, &L.d_gu));
        RCHECK(build_dense(m, {p + "ff.w_out"}, {D}, m->ff, &L.d_down));
        if (c.quant_type == 2)
            for (DenseLin* dl : {&L.d_qkv, &L.d_o, &L.d_gu, &L.d_down}) RCHECK(dense_to_int8(m, dl));
    }
    return ZL_OK;
}

int finalize_globals(zl_llama* m) {
    const auto& c = m->cfg;
    RCHECK(take_vector(m, "token_embedding.weight", c.vocab_size * c.dim_model, &m->emb));
    m->weight_bytes -= (double)c.vocab_size * c.dim_model * 2;   // the embedding table is gathered, not streamed
    RCHECK(take_vector(m, "output_layernorm.weight", c.dim_model, &m->ln_f));
    if (find(m, "lm_head.weight")) {
        RCHECK(take_vector(m, "lm_head.weight", m->vshard * c.dim_model, &m->lm_head));   // vocab-parallel shard
    } else {
        ZL_CHECK_SUPPORTED(c.tp_size == 1);   // tied lm_head is only wired for a single rank
        m->lm_head = m->emb;   // tied (Llama-3.2-1B)
        m->lm_head_tied = true;
        m->weight_bytes += (double)c.vocab_size * c.dim_model * 2;
    }
    return ZL_OK;
}

// the parameters of a task without sampling state: zl_sample then picks exactly what zl_argmax picks
constexpr zl_sample_params_t kGreedyParams = {1.0f, 1.0f, 1.0f, 0.0f, 0, 0};

// stream-ordered: parameters to the device, seen set and draw counter cleared
int write_sampling(zl_llama* m, int task, const zl_sample_params_t& p) {
    const size_t words = (size_t)(m->vshard + 31) / 32;
    ZL_CHECK_CUDA(cudaMemcpyAsync(m->d_sparams + task, &p, sizeof(p), cudaMemcpyHostToDevice, m->stream));
    ZL_CHECK_CUDA(cudaMemsetAsync(m->d_seen + task * words, 0, words * sizeof(uint32_t), m->stream));
    ZL_CHECK_CUDA(cudaMemsetAsync(m->d_draws + task, 0, sizeof(uint32_t), m->stream));
    return ZL_OK;
}

int alloc_runtime(zl_llama* m) {
    const auto& c = m->cfg;
    const int B = c.max_batch, D = c.dim_model, d = c.dim_head;
    const size_t kv_task = (size_t)c.max_seq * m->hkv * d * 2;
    for (auto& L : m->layers) {
        RCHECK(dmalloc(&L.kbuf, kv_task * B));
        RCHECK(dmalloc(&L.vbuf, kv_task * B));
        // never-written rows must be finite: masked keys still multiply their V rows by an exact 0, and with the
        // dual-stream prefill one half's attention sees the other half's rows before they are appended
        ZL_CHECK_CUDA(cudaMemsetAsync(L.kbuf, 0, kv_task * B, m->stream));
        ZL_CHECK_CUDA(cudaMemsetAsync(L.vbuf, 0, kv_task * B, m->stream));
        RCHECK(dmalloc((void**)&L.k_addrs, sizeof(void*) * B));
        RCHECK(dmalloc((void**)&L.v_addrs, sizeof(void*) * B));
        k_ptr_table<<<cdiv(B, 256), 256, 0, m->stream>>>(L.k_addrs, (char*)L.kbuf, kv_task, B);
        k_ptr_table<<<cdiv(B, 256), 256, 0, m->stream>>>(L.v_addrs, (char*)L.vbuf, kv_task, B);
        ZL_CHECK_LAUNCH();
    }
    const int T = c.prefill_chunk > B ? c.prefill_chunk : B;   // tokens per launch: decode batch or prefill chunk
    m->tok_cap = T;
    RCHECK(dmalloc(&m->h, (size_t)T * D * 2));
    RCHECK(dmalloc(&m->xn, (size_t)T * D * 2));
    if (c.tp_size > 1) RCHECK(dmalloc(&m->h2, (size_t)T * D * 2));
    RCHECK(dmalloc(&m->pend, (size_t)T * D * 2));
    RCHECK(dmalloc(&m->qkv, (size_t)T * (m->hq + 2 * m->hkv) * d * 2));
    RCHECK(dmalloc(&m->q, (size_t)T * m->hq * d * 2));
    RCHECK(dmalloc(&m->ao, (size_t)T * m->hq * d * 2));
    RCHECK(dmalloc(&m->gu, (size_t)T * 2 * m->ff * 2));
    RCHECK(dmalloc(&m->act, (size_t)T * m->ff * 2));
    RCHECK(dmalloc((void**)&m->logits, (size_t)B * c.vocab_size * 4));
    RCHECK(dmalloc(&m->cand, (size_t)((B * 8 + 15) / 16) * 16));
    RCHECK(dmalloc(&m->cand_all, (size_t)((B * 8 + 15) / 16) * 16 * c.tp_size));
    RCHECK(dmalloc((void**)&m->cosb, (size_t)T * d * 4));
    RCHECK(dmalloc((void**)&m->sinb, (size_t)T * d * 4));
    RCHECK(dmalloc((void**)&m->d_tokens, B * 4));
    RCHECK(dmalloc((void**)&m->d_pos, B * 4));
    RCHECK(dmalloc((void**)&m->d_lens, B * 4));
    if (c.quant_type == 2 || c.quant_type == 7) {
        int kmax = D > m->ff ? D : m->ff;
        kmax = kmax > m->hq * d ? kmax : m->hq * d;
        RCHECK(dmalloc(&m->xq, (size_t)T * kmax));
        RCHECK(dmalloc((void**)&m->xs, (size_t)T * 4));
    }
    if (c.prefill_chunk > 0) {
        RCHECK(dmalloc((void**)&m->d_tb, T * 4));
        RCHECK(dmalloc((void**)&m->d_pf_tokens, T * 4));
        RCHECK(dmalloc((void**)&m->d_pf_pos, T * 4));
        RCHECK(dmalloc((void**)&m->d_mask, (size_t)c.prefill_chunk * c.max_seq));
    }
    RCHECK(dmalloc((void**)&m->d_next, B * 4));
    RCHECK(dmalloc((void**)&m->d_iota, B * 4));
    k_iota<<<cdiv(B, 256), 256, 0, m->stream>>>(m->d_iota, B);
    ZL_CHECK_LAUNCH();
    m->attn_ws_bytes = zl_decode_attention_workspace_bytes(T, 1, m->hq, d, c.max_seq);
    RCHECK(dmalloc(&m->attn_ws, m->attn_ws_bytes));
    RCHECK(dmalloc(&m->argmax_ws, zl_argmax_workspace_bytes(B)));
    RCHECK(dmalloc((void**)&m->d_sparams, sizeof(zl_sample_params_t) * B));
    RCHECK(dmalloc((void**)&m->d_seen, sizeof(uint32_t) * B * (size_t)((m->vshard + 31) / 32)));
    RCHECK(dmalloc((void**)&m->d_draws, sizeof(uint32_t) * B));
    m->sampling.assign(B, 0);
    for (int t = 0; t < B; ++t) RCHECK(write_sampling(m, t, kGreedyParams));
    ZL_CHECK_CUDA(cudaMallocHost((void**)&m->h_stage, sizeof(int32_t) * (4 * B + 4 + T)));
    ZL_CHECK_CUDA(cudaMallocHost((void**)&m->h_ring, sizeof(int32_t) * zl_llama::kStageSlots * 2 * B));
    for (int i = 0; i < zl_llama::kStageSlots; ++i)
        ZL_CHECK_CUDA(cudaEventCreateWithFlags(&m->ring_ev[i], cudaEventDisableTiming));
    ZL_CHECK_CUDA(cudaStreamSynchronize(m->stream));
    return ZL_OK;
}

// The decode-step kernel chain (captured into a graph by run_step).
// cfg.fuse: 0 = one kernel per reference operator; 1 = RMSNorm folded into the following W4 GEMM;
//           2 = additionally qkv split + RoPE + KV append folded into the qkv GEMM epilogue.
// cap of the L2 prefetch a kernel issues for its successor (bytes); ZL_L2_PREFETCH_MB overrides, 0 disables
static size_t prefetch_cap() {
    static long v = -1;
    if (v < 0) {
        const char* e = getenv("ZL_L2_PREFETCH_MB");
        v = e ? atol(e) : 0;   // measured on B200: bulk L2 prefetch competes with the ring's TMA traffic; off by default
    }
    return (size_t)v << 20;
}
// which blob each kernel of a layer prefetches (ZL_L2_PREFETCH_PLAN, 5 digits for qkv,attn(unused),o,gate_up,down ->
// 0 none, 1 o, 2 gate_up, 3 down, 4 next qkv); experiment knob, only read when ZL_L2_PREFETCH_MB > 0
static int prefetch_plan(int slot) {
    static int plan[5] = {-1, 0, 0, 0, 0};
    if (plan[0] < 0) {
        const char* e = getenv("ZL_L2_PREFETCH_PLAN");
        const char* d = (e && strlen(e) == 5) ? e : "10234";
        for (int i = 0; i < 5; ++i) plan[i] = d[i] - '0';
    }
    return plan[slot];
}

// resolve the plan entry of kernel `slot` (0 qkv, 1 attention, 2 o, 3 gate_up, 4 down) of layer l to a packed blob
static void prefetch_target(zl_llama* m, int l, int slot, int B, const void** ptr, size_t* bytes) {
    *ptr = nullptr;
    *bytes = 0;
    const auto& c = m->cfg;
    if (!(c.quant_type == 5 || c.quant_type == 6) || prefetch_cap() == 0) return;
    const int what = prefetch_plan(slot);
    const W4Lin* t = nullptr;
    Layer& L = m->layers[l];
    if (what == 1) t = &L.q_o;
    else if (what == 2) t = &L.q_gu;
    else if (what == 3) t = &L.q_down;
    else if (what == 4 && l + 1 < c.num_layers) t = &m->layers[l + 1].q_qkv;
    if (!t) return;
    const bool t_int = t->packed_i && !getenv("ZL_W4_FORCE_HALF") && zl_w4_int_layout_route(B, t->N, t->K) != 0;
    *ptr = t_int ? t->packed_i : t->packed;
    const size_t nb = zl_w4_packed_bytes(t->N, t->K, c.group_size);
    *bytes = nb < prefetch_cap() ? nb : prefetch_cap();
}

// ZL_NO_PDL_MASK (experiments): launch these kernels with a full dependency instead of a programmatic one.
// 1 qkv GEMM, 2 attention, 4 o GEMM, 8 gate_up GEMM, 16 down GEMM, 32 final norm, 64 lm_head, 128 argmax.
// Default 70 = lm_head + o GEMM + attention: a PDL-launched lm_head measured 128 us slower per step than a normally
// launched one (tools/gpu_tail.sh); early-launched o GEMM / attention CTAs cost another ~1 % each.
static int no_pdl_mask(bool tensor_parallel = false) {
    static int v = -2;
    if (v == -2) {
        const char* e = getenv("ZL_NO_PDL_MASK");
        v = e ? atoi(e) : -1;
    }
    if (v >= 0) return v;
    // single GPU: lm_head, o GEMM, attention with full dependencies measured best (tools/gpu_pdlmask.sh: 640 -> 710 tok/s);
    // tensor parallel (exchange inside the GEMMs): a PDL-launched attention kernel wins (N = 2: 783 vs 754 tok/s, r2s)
    return tensor_parallel ? 68 : 70;
}

int w4_gemm(zl_llama* m, const void* x, int ldx, const W4Lin& w, const void* residual, void* y, int B, int epi,
            const void* ln_w, const Layer* rope_layer, int layer = -1, int slot = -1, int row0 = 0, int force_no_pdl = 0,
            int tp_mode = 0, void* tp_h_out = nullptr, int tp_index = 0) {
    const auto& c = m->cfg;
    zl_w4_fused_args_t a = {};
    a.x = x;
    a.ldx = ldx;
    const int route = (w.packed_i && !getenv("ZL_W4_FORCE_HALF")) ? zl_w4_int_layout_route(B, w.N, w.K) : 0;
    const bool use_int = route != 0;
    a.packed = use_int ? w.packed_i : w.packed;
    a.variant = use_int ? 1 : 0;
    if (route == 4 && ln_w) {
        // the tcgen05 kernel reads x through the TMA engine: the RMSNorm runs as its own kernel (reference order,
        // block.cpp:125,131) into the matching rows of xn
        const size_t off = (const char*)x - (const char*)m->h;
        void* xn = (char*)m->xn + off;
        RCHECK(zl_rmsnorm(x, ln_w, xn, B, w.K, c.eps, 1.f, c.dtype, force_no_pdl ? 0 : c.use_pdl, m->stream));
        a.x = xn;
        ln_w = nullptr;
    }
    if (layer >= 0) {
        size_t nb = 0;
        prefetch_target(m, layer, slot, B, &a.prefetch_ptr, &nb);
        a.prefetch_bytes = nb;
    }
    if (!a.packed) {
        zl_set_last_error(__FILE__, __LINE__, "no packed weight variant for this batch size");
        return ZL_ERR_STATE;
    }
    a.bias = w.bias;
    a.residual = residual;
    a.y = y;
    a.M = B;
    a.N = w.N;
    a.K = w.K;
    a.group_size = c.group_size;
    a.epilogue = epi;
    {
        const int bit = slot == 0 ? 1 : slot == 2 ? 4 : slot == 3 ? 8 : slot == 4 ? 16 : 0;
        a.pdl = (no_pdl_mask(c.tp_size > 1) & bit) ? 0 : c.use_pdl;
    }
    a.ln_weight = ln_w;
    a.eps = c.eps;
    if (rope_layer) {
        // row0: first token row of this call inside the step's activation matrices (dual-stream prefill halves)
        a.cos = m->cosb + (size_t)row0 * c.dim_head;
        a.sin = m->sinb + (size_t)row0 * c.dim_head;
        a.q_out = (char*)m->q + (size_t)row0 * m->hq * c.dim_head * 2;
        a.token_batch = m->cur_tb + row0;
        a.placement = m->cur_pos + row0;
        a.k_addrs = rope_layer->k_addrs;
        a.v_addrs = rope_layer->v_addrs;
        a.num_heads = m->hq;
        a.num_kv_heads = m->hkv;
        a.dim_head = c.dim_head;
    }
    if (force_no_pdl) a.pdl = 0;
    if (tp_mode) {
        a.tp_comm = m->comm;
        a.tp_mode = tp_mode;
        a.tp_h_out = tp_h_out;
        a.tp_index = tp_index;
    }
    return zl_w4a16_gemm_fused(&a, m->stream);
}

static int num_sms() { return device_sm_count(); }

// ZL_DEBUG_SKIP (bit mask, timing experiments only -- results are wrong when set):
// 1 attention, 2 qkv GEMM, 4 o GEMM, 8 gate/up GEMM, 16 down GEMM, 32 lm_head, 64 rope/append kernel
static int debug_skip() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("ZL_DEBUG_SKIP");
        v = e ? atoi(e) : 0;
    }
    return v;
}

// One non-W4 Linear of the decode chain: dense (NormalLinear), or W8A8 = activation quant + fused 8-bit GEMM
// (Int8Linear::forward / Fp8Linear::forward in two launches instead of three).
int dense_or_w8(zl_llama* m, const void* x, const DenseLin& L, void* y, int B, int pdl) {
    const auto& c = m->cfg;
    cudaStream_t st = m->stream;
    if (!L.w8) return zl_dense_gemm_skinny(x, L.K, L.w, L.bias, y, B, L.N, L.K, c.dtype, c.dtype, pdl, st);
    if (L.w8_kind == ZL_W8_INT8) {
        RCHECK(zl_int8_quant_per_token(x, L.K, m->xq, m->xs, B, L.K, c.dtype, pdl, st));
        return zl_w8a8_gemm(m->xq, m->xs, L.w8, L.w_scale, c.dtype, L.bias, y, B, L.N, L.K, ZL_W8_INT8, c.dtype, pdl, st);
    }
    RCHECK(zl_fp8_quant_per_tensor(x, m->xq, m->xs, (size_t)B * L.K, c.dtype, pdl, st));
    return zl_w8a8_gemm(m->xq, m->xs, L.w8, L.w_scale, ZL_F32, L.bias, y, B, L.N, L.K, ZL_W8_FP8_ROWS, c.dtype, pdl, st);
}

// pf != nullptr: one chunk of a prompt (tokens of ONE task at consecutive positions) instead of one token per task
struct PrefillChunk {
    int task, pos0, n;
    bool last;   // run final norm + lm_head + pick on the chunk's last token
};

// ------------------------------------------------------------------------------------------------------------------
// Dual-stream chunked prefill of a W4 model (EncoderLayer::impl::dual_stream_encode, src/nn/block/block.cpp:205-441):
// the chunk's tokens are split in two halves that walk the layers as a 2-stage pipeline -- while the reduce stream
// combines half A's row-parallel partial sums (NVLink all-reduce fused with the residual add; a plain residual add when
// tp_size == 1), the compute stream already runs half B's GEMMs / attention.  The reference creates its second stream
// and 2*num_split events on every forward (block.cpp:220-224, 260-267); here they live in the model object.
//   compute: S1(h0) S1(h1) S3(h0) S3(h1) | next layer ...      S1 = qkv(+RoPE, KV append) -> attention -> o GEMM
//   reduce :        R1(h0) R1(h1) R2(h0) R2(h1)                S3 = gate_up (SwiGLU) -> down GEMM ; R = reduce + residual
// ------------------------------------------------------------------------------------------------------------------
int ensure_dual_resources(zl_llama* m) {
    if (m->reduce_stream) return ZL_OK;
    ZL_CHECK_CUDA(cudaStreamCreateWithFlags(&m->reduce_stream, cudaStreamNonBlocking));
    for (int h = 0; h < 2; ++h)
        for (cudaEvent_t* e : {&m->ev_o[h], &m->ev_r1[h], &m->ev_dn[h], &m->ev_r2[h]})
            ZL_CHECK_CUDA(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
    return ZL_OK;
}

static bool prefill_dual_enabled(const zl_llama* m, int n) {
    // ZL_PREFILL_DUAL: 0 never, 1 always (on one GPU the "reduce" is the residual add: exercises the pipeline),
    // 2 (default) = when tensor parallel.  Read per call: prefill is not a latency-critical path.
    const char* e = getenv("ZL_PREFILL_DUAL");
    const int force = e ? atoi(e) : 2;
    const auto& c = m->cfg;
    if (!(c.quant_type == 5 || c.quant_type == 6) || c.fuse < 1 || n < 16) return false;
    return force == 1 || (force == 2 && c.tp_size > 1);
}

int prefill_layers_dual(zl_llama* m, const PrefillChunk& pf) {
    const auto& c = m->cfg;
    RCHECK(ensure_dual_resources(m));
    const int D = c.dim_model, d = c.dim_head, dt = c.dtype;
    const bool tp = c.tp_size > 1;
    cudaStream_t cs = m->stream, rs = m->reduce_stream;
    const float scale = 1.0f / sqrtf((float)d);
    const int n0 = (pf.n / 2 + 7) / 8 * 8 < pf.n ? (pf.n / 2 + 7) / 8 * 8 : pf.n / 2;   // rows of half 0
    const int r0[2] = {0, n0}, nh[2] = {n0, pf.n - n0};
    const int len_buf = pf.pos0 + pf.n;
    auto rows = [&](void* base, int row, size_t row_bytes) { return (char*)base + (size_t)row * row_bytes; };
    auto reduce = [&](int h) -> int {   // h rows: h += sum over ranks of pend
        void* hp = rows(m->h, r0[h], (size_t)D * 2);
        void* pp = rows(m->pend, r0[h], (size_t)D * 2);
        if (tp) return zl_allreduce_one_shot(m->comm, pp, hp, hp, (size_t)nh[h] * D, dt, c.tp_int8, 0, rs);
        return zl_element_add_scale(hp, pp, hp, (size_t)nh[h] * D, 1.0f, dt, rs);
    };
    for (int l = 0; l < c.num_layers; ++l) {
        Layer& L = m->layers[l];
        for (int h = 0; h < 2; ++h) {   // S1
            if (l > 0) ZL_CHECK_CUDA(cudaStreamWaitEvent(cs, m->ev_r2[h], 0));
            void* hp = rows(m->h, r0[h], (size_t)D * 2);
            if (c.fuse >= 2) {
                RCHECK(w4_gemm(m, hp, D, L.q_qkv, nullptr, nullptr, nh[h], ZL_EPI_QKV_ROPE, L.ln_attn, &L, -1, -1, r0[h], 1));
            } else {
                void* qp = rows(m->qkv, r0[h], (size_t)(m->hq + 2 * m->hkv) * d * 2);
                RCHECK(w4_gemm(m, hp, D, L.q_qkv, nullptr, qp, nh[h], ZL_EPI_NONE, L.ln_attn, nullptr, -1, -1, 0, 1));
                RCHECK(zl_qkv_rope_append(m->cosb + (size_t)r0[h] * d, m->sinb + (size_t)r0[h] * d, qp,
                                          rows(m->q, r0[h], (size_t)m->hq * d * 2), m->cur_tb + r0[h], m->cur_pos + r0[h],
                                          L.k_addrs, L.v_addrs, nh[h], m->hq, m->hkv, d, 1, 1, m->d_lens, dt, 0, cs));
            }
            // causal rows r0.. of the chunk's mask; keys of BOTH halves are visible as far as the mask allows, so half 1
            // needs half 0's K/V rows, which the same stream appended just before
            RCHECK(zl_decode_attention(rows(m->q, r0[h], (size_t)m->hq * d * 2), m->d_lens + pf.task, L.k_addrs + pf.task,
                                       L.v_addrs + pf.task, m->d_mask + (size_t)r0[h] * len_buf, scale, len_buf,
                                       rows(m->ao, r0[h], (size_t)m->hq * d * 2), 1, nh[h], m->hq, m->hkv, d, 1, m->attn_ws,
                                       m->attn_ws_bytes, dt, 0, cs));
            RCHECK(w4_gemm(m, rows(m->ao, r0[h], (size_t)m->hq * d * 2), m->hq * d, L.q_o, nullptr,
                           rows(m->pend, r0[h], (size_t)D * 2), nh[h], ZL_EPI_NONE, nullptr, nullptr, -1, -1, 0, 1));
            ZL_CHECK_CUDA(cudaEventRecord(m->ev_o[h], cs));
            ZL_CHECK_CUDA(cudaStreamWaitEvent(rs, m->ev_o[h], 0));   // R1
            RCHECK(reduce(h));
            ZL_CHECK_CUDA(cudaEventRecord(m->ev_r1[h], rs));
        }
        for (int h = 0; h < 2; ++h) {   // S3
            ZL_CHECK_CUDA(cudaStreamWaitEvent(cs, m->ev_r1[h], 0));
            void* hp = rows(m->h, r0[h], (size_t)D * 2);
            void* ap = rows(m->act, r0[h], (size_t)m->ff * 2);
            RCHECK(w4_gemm(m, hp, D, L.q_gu, nullptr, ap, nh[h], ZL_EPI_SWIGLU, L.ln_ff, nullptr, -1, -1, 0, 1));
            RCHECK(w4_gemm(m, ap, m->ff, L.q_down, nullptr, rows(m->pend, r0[h], (size_t)D * 2), nh[h], ZL_EPI_NONE, nullptr,
                           nullptr, -1, -1, 0, 1));
            ZL_CHECK_CUDA(cudaEventRecord(m->ev_dn[h], cs));
            ZL_CHECK_CUDA(cudaStreamWaitEvent(rs, m->ev_dn[h], 0));   // R2
            RCHECK(reduce(h));
            ZL_CHECK_CUDA(cudaEventRecord(m->ev_r2[h], rs));
        }
    }
    for (int h = 0; h < 2; ++h) ZL_CHECK_CUDA(cudaStreamWaitEvent(cs, m->ev_r2[h], 0));
    return ZL_OK;
}

// does the launch sequence for decode tasks 0..n_tasks-1 (or the prefilled task) pick with zl_sample?
bool step_samples(const zl_llama* m, int n_tasks, const PrefillChunk* pf) {
    if (pf) return m->sampling[pf->task] != 0;
    for (int t = 0; t < n_tasks; ++t)
        if (m->sampling[t]) return true;
    return false;
}

int enqueue_step(zl_llama* m, int n_tasks, int len_bucket, const PrefillChunk* pf = nullptr) {
    const auto& c = m->cfg;
    const int B = pf ? pf->n : n_tasks;   // rows (tokens) of every activation matrix in this launch sequence
    const int skip = debug_skip();
    const int D = c.dim_model, d = c.dim_head, dt = c.dtype, pdl = c.use_pdl;
    const int npm = no_pdl_mask(c.tp_size > 1);
    auto P = [&](int bit) { return (npm & bit) ? 0 : pdl; };
    cudaStream_t st = m->stream;
    const bool w4 = c.quant_type == 5 || c.quant_type == 6;
    const bool tp = c.tp_size > 1;
    if (tp && !m->comm) {
        zl_set_last_error(__FILE__, __LINE__, "tp_size > 1 but zl_llama_set_comm was not called");
        return ZL_ERR_STATE;
    }
    const float scale = 1.0f / sqrtf((float)d);   // attention.cpp:89

    if (pf) {
        k_prefill_setup<<<8, 256, 0, st>>>(m->d_pf_pos, m->d_tb, m->d_lens, m->d_mask, pf->task, pf->pos0, pf->n);
        ZL_CHECK_LAUNCH();
    } else {
        ZL_CHECK_CUDA(launch(k_lens_from_pos, dim3(cdiv(B, 64)), dim3(64), 0, st, false, (const int32_t*)m->d_pos,
                             m->d_lens, B, g_w4_trace));
    }
    m->cur_tb = pf ? m->d_tb : m->d_iota;
    m->cur_pos = pf ? m->d_pf_pos : m->d_pos;
    m->cur_tokens = pf ? m->d_pf_tokens : m->d_tokens;
    RCHECK(zl_rope_cos_sin(m->cur_pos, m->cosb, m->sinb, B, d, c.rope_theta, c.rope_llama3_factor,
                           c.rope_low_freq_factor, c.rope_high_freq_factor, c.rope_orig_ctx, 1, st));
    RCHECK(zl_embedding(m->cur_tokens, m->emb, m->h, B, D, c.vocab_size, dt, 0, st));
    const bool dual = pf && prefill_dual_enabled(m, pf->n);
    if (dual) RCHECK(prefill_layers_dual(m, *pf));
    // Tensor parallel, decode-sized launches of a W4 model: the exchange rides inside the GEMMs.  The row-parallel GEMMs
    // (o_proj, w_out) push their fp16 partial tiles into every rank's inbox from the epilogue; the next GEMM (gate_up, next
    // layer's qkv) reduces them in rank order while it stages its activations and writes the new residual stream to the
    // other of the two buffers h / h2.  Only the last layer's w_out keeps the stand-alone one-shot kernel (the final norm
    // is not a GEMM).  ZL_TP_UNFUSED=1 keeps the separate exchange kernels everywhere (A/B).
    bool tp_fused = tp && w4 && !pf && c.fuse >= 1 && !c.tp_int8 && dt == ZL_F16 && !getenv("ZL_TP_UNFUSED") && !skip &&
                    (size_t)B * D * 2 <= zl_comm_slot_bytes(m->comm) && 2 * c.num_layers <= 512;
    if (tp_fused) {
        const Layer& L0 = m->layers[0];
        for (const W4Lin* w : {&L0.q_qkv, &L0.q_o, &L0.q_gu, &L0.q_down})
            if (!w->packed_i || zl_w4_int_layout_route(B, w->N, w->K) != 3) tp_fused = false;
    }
    if (tp_fused) RCHECK(zl_comm_ll_begin_step(m->comm, st));   // the word tags of this step's exchanges
    void* hc = m->h;    // current residual stream
    void* ho = m->h2;   // where the next fused reduce-in writes it
    bool pending = false;   // partial sums of the previous row-parallel GEMM are in flight to the inboxes
    int xi = 0;             // index of the next exchange of the step (producer and consumer use the same one)
    const int xodd = ((2 * c.num_layers - 1) & 1) << 9;   // 2 L - 1 exchanges per step: odd -> bit 9 of tp_index
    for (int l = 0; l < (dual ? 0 : c.num_layers); ++l) {
        Layer& L = m->layers[l];
        if (w4) {
            const void* xin = m->xn;
            const void* lnw = nullptr;
            if (c.fuse >= 1) {
                xin = hc;
                lnw = L.ln_attn;
            } else {
                RCHECK(zl_rmsnorm(hc, L.ln_attn, m->xn, B, D, c.eps, 1.f, dt, pdl, st));
            }
            const int tpm = pending ? 1 : 0;
            if (skip & 2) {
            } else if (c.fuse >= 2) {
                RCHECK(w4_gemm(m, xin, D, L.q_qkv, nullptr, nullptr, B, ZL_EPI_QKV_ROPE, lnw, &L, l, 0, 0, 0, tpm, ho, (xi - 1) | xodd));
            } else {
                RCHECK(w4_gemm(m, xin, D, L.q_qkv, nullptr, m->qkv, B, ZL_EPI_NONE, lnw, nullptr, l, 0, 0, 0, tpm, ho, (xi - 1) | xodd));
            }
            if (pending) {
                std::swap(hc, ho);
                pending = false;
            }
        } else {
            // residual of the previous layer's FFN is folded into this norm (block.cpp:139-141 + 131)
            RCHECK(zl_add_rmsnorm(m->h, l == 0 ? nullptr : m->pend, L.ln_attn, m->h, m->xn, B, D, c.eps, 1.f, 0, dt,
                                  pdl, st));
            RCHECK(dense_or_w8(m, m->xn, L.d_qkv, m->qkv, B, pdl));
        }
        if (!(w4 && c.fuse >= 2) && !(skip & 64))
            RCHECK(zl_qkv_rope_append(m->cosb, m->sinb, m->qkv, m->q, m->cur_tb, m->cur_pos, L.k_addrs, L.v_addrs, B,
                                      m->hq, m->hkv, d, 1, 1, m->d_lens, dt, pdl, st));
        if (!(skip & 1)) {
            const void* pfp = nullptr;
            size_t pfb = 0;
            prefetch_target(m, l, 1, B, &pfp, &pfb);
            zl_decode_attention_set_prefetch(pfp, pfb);
        }
        if (pf) {
            // one task, len_q = chunk, causal int8 mask (Attention::dynamic_batch_forward with len_q > 1, attention.cpp:846-964)
            RCHECK(zl_decode_attention(m->q, m->d_lens + pf->task, L.k_addrs + pf->task, L.v_addrs + pf->task, m->d_mask,
                                       scale, pf->pos0 + pf->n, m->ao, 1, pf->n, m->hq, m->hkv, d, 1, m->attn_ws,
                                       m->attn_ws_bytes, dt, pdl, st));
        } else if (!(skip & 1))
            RCHECK(zl_decode_attention(m->q, m->d_lens, L.k_addrs, L.v_addrs, nullptr, scale, len_bucket, m->ao, B, 1,
                                       m->hq, m->hkv, d, 1, m->attn_ws, m->attn_ws_bytes, dt, P(2), st));
        if (w4) {
            if (skip & 4) {
            } else if (tp_fused) {
                RCHECK(w4_gemm(m, m->ao, m->hq * d, L.q_o, nullptr, nullptr, B, ZL_EPI_NONE, nullptr, nullptr, l, 2, 0, 0, 2, nullptr, (xi++) | xodd));
                pending = true;
            } else if (tp) {
                // row-parallel: partial sums -> one-shot NVLink all-reduce fused with the residual add
                RCHECK(w4_gemm(m, m->ao, m->hq * d, L.q_o, nullptr, m->pend, B, ZL_EPI_NONE, nullptr, nullptr, l, 2));
                RCHECK(zl_allreduce_one_shot(m->comm, m->pend, hc, hc, (size_t)B * D, dt, c.tp_int8, pdl, st));
            } else {
                RCHECK(w4_gemm(m, m->ao, m->hq * d, L.q_o, hc, hc, B, ZL_EPI_RESIDUAL, nullptr, nullptr, l, 2));
            }
            const void* xin = m->xn;
            const void* lnw = nullptr;
            if (c.fuse >= 1) {
                xin = hc;
                lnw = L.ln_ff;
            } else {
                RCHECK(zl_rmsnorm(hc, L.ln_ff, m->xn, B, D, c.eps, 1.f, dt, pdl, st));
            }
            if (!(skip & 8))
                RCHECK(w4_gemm(m, xin, D, L.q_gu, nullptr, m->act, B, ZL_EPI_SWIGLU, lnw, nullptr, l, 3, 0, 0, pending ? 1 : 0, ho, (xi - 1) | xodd));
            if (pending) {
                std::swap(hc, ho);
                pending = false;
            }
            if (skip & 16) {
            } else if (tp_fused && l + 1 < c.num_layers) {
                RCHECK(w4_gemm(m, m->act, m->ff, L.q_down, nullptr, nullptr, B, ZL_EPI_NONE, nullptr, nullptr, l, 4, 0, 0, 2, nullptr, (xi++) | xodd));
                pending = true;
            } else if (tp) {
                RCHECK(w4_gemm(m, m->act, m->ff, L.q_down, nullptr, m->pend, B, ZL_EPI_NONE, nullptr, nullptr, l, 4));
                RCHECK(zl_allreduce_one_shot(m->comm, m->pend, hc, hc, (size_t)B * D, dt, c.tp_int8, pdl, st));
            } else {
                RCHECK(w4_gemm(m, m->act, m->ff, L.q_down, hc, hc, B, ZL_EPI_RESIDUAL, nullptr, nullptr, l, 4));
            }
        } else {
            RCHECK(dense_or_w8(m, m->ao, L.d_o, m->pend, B, pdl));
            if (tp) RCHECK(zl_allreduce_one_shot(m->comm, m->pend, nullptr, m->pend, (size_t)B * D, dt, c.tp_int8, pdl, st));
            RCHECK(zl_add_rmsnorm(m->h, m->pend, L.ln_ff, m->h, m->xn, B, D, c.eps, 1.f, 0, dt, pdl, st));
            RCHECK(dense_or_w8(m, m->xn, L.d_gu, m->gu, B, pdl));
            RCHECK(zl_gate_mul(m->gu, 2 * m->ff, (char*)m->gu + (size_t)m->ff * 2, 2 * m->ff, m->act, m->ff, B,
                               m->ff, 0, dt, st));
            RCHECK(dense_or_w8(m, m->act, L.d_down, m->pend, B, pdl));
            if (tp) RCHECK(zl_allreduce_one_shot(m->comm, m->pend, nullptr, m->pend, (size_t)B * D, dt, c.tp_int8, pdl, st));
        }
    }
    if (pf) {
        if (!pf->last) return ZL_OK;
        // only the last prompt position feeds the head: move it to row 0 semantics by pointing at its row
        const size_t off = (size_t)(pf->n - 1) * D * 2;
        if (w4) {
            RCHECK(zl_rmsnorm((char*)m->h + off, m->ln_f, m->xn, 1, D, c.eps, 1.f, dt, pdl, st));
        } else {
            RCHECK(zl_add_rmsnorm((char*)m->h + off, (char*)m->pend + off, m->ln_f, (char*)m->h + off, m->xn, 1, D, c.eps,
                                  1.f, 0, dt, pdl, st));
        }
    } else if (w4) {
        RCHECK(zl_rmsnorm(hc, m->ln_f, m->xn, B, D, c.eps, 1.f, dt, P(32), st));
    } else {
        RCHECK(zl_add_rmsnorm(m->h, m->pend, m->ln_f, m->h, m->xn, B, D, c.eps, 1.f, 0, dt, P(32), st));
    }
    const int HB = pf ? 1 : B;   // rows that reach lm_head
    // vocab-parallel lm_head (embedding.cu:353-392): each rank owns vshard rows
    if (!(skip & 32))
        RCHECK(zl_dense_gemm_skinny(m->xn, D, m->lm_head, nullptr, m->logits, HB, m->vshard, D, dt, ZL_F32, P(64), st));
    if (step_samples(m, n_tasks, pf)) {
        // row 0 of a prefill belongs to pf->task: d_iota[task] == task
        RCHECK(zl_sample(m->logits, HB, m->vshard, pf ? m->d_iota + pf->task : m->d_iota, m->d_sparams, m->d_seen,
                         m->d_draws, m->d_next, nullptr, 0, P(128), st));
    } else if (!tp) {
        RCHECK(zl_argmax(m->logits, m->d_next, HB, m->vshard, m->argmax_ws, zl_argmax_workspace_bytes(HB), P(128), st));
    } else {
        // instead of all-gathering (B, V) logits, exchange one {value, index} candidate per token
        const int stride = ((HB * 8 + 15) / 16) * 2;   // int2 records per rank slot (16-byte multiple)
        RCHECK(zl_argmax_candidates(m->logits, m->cand, HB, m->vshard, c.tp_rank * m->vshard, m->argmax_ws,
                                    zl_argmax_workspace_bytes(HB), pdl, st));
        RCHECK(zl_allgather_small(m->comm, m->cand, m->cand_all, (size_t)stride * 8, pdl, st));
        RCHECK(zl_argmax_merge(m->cand_all, m->d_next, HB, c.tp_size, stride, pdl, st));
    }
    return ZL_OK;
}

// attention split counts are baked into the graph: one graph per (batch, length bucket)
int len_bucket_of(const zl_llama* m, int max_len) {
    int b = 256;
    while (b < max_len) b <<= 1;
    return b < m->cfg.max_seq ? b : (m->cfg.max_seq > 256 ? m->cfg.max_seq : 256);
}

int run_step(zl_llama* m, int B) {
    const int bucket = len_bucket_of(m, m->cur_max_len);
    if (!m->cfg.use_graph) return enqueue_step(m, B, bucket);
    // sampling steps have a graph of their own: batches without a sampling task replay exactly the greedy graph
    const long long key = ((long long)B << 33) | ((long long)step_samples(m, B, nullptr) << 32) | (unsigned)bucket;
    auto it = m->graphs.find(key);
    if (it == m->graphs.end()) {
        cudaGraph_t graph = nullptr;
        ZL_CHECK_CUDA(cudaStreamBeginCapture(m->stream, cudaStreamCaptureModeThreadLocal));
        int rc = enqueue_step(m, B, bucket);
        cudaError_t ce = cudaStreamEndCapture(m->stream, &graph);
        if (rc != ZL_OK) {
            if (graph) cudaGraphDestroy(graph);
            return rc;
        }
        ZL_CHECK_CUDA(ce);
        cudaGraphExec_t exec = nullptr;
        ZL_CHECK_CUDA(cudaGraphInstantiate(&exec, graph, 0));
        size_t n_nodes = 0;
        cudaGraphGetNodes(graph, nullptr, &n_nodes);
        m->kernels_per_step = (int)n_nodes;
        cudaGraphDestroy(graph);
        it = m->graphs.emplace(key, exec).first;
    }
    ZL_CHECK_CUDA(cudaGraphLaunch(it->second, m->stream));
    return ZL_OK;
}

}  // namespace

extern "C" int zl_llama_create(const zl_llama_config_t* cfg, zl_llama_t** out) {
    ZL_CHECK_ARG(cfg && out);
    ZL_CHECK_ARG(cfg->num_layers > 0 && cfg->dim_model > 0 && cfg->num_heads > 0 && cfg->num_kv_heads > 0);
    ZL_CHECK_ARG(cfg->dim_head > 0 && cfg->dim_ff > 0 && cfg->vocab_size > 0 && cfg->max_batch > 0 &&
                 cfg->max_seq > 0);
    // QuantType 8 (GPTQ_Marlin, linear.cpp:1247-1451) loads the same GPTQ checkpoint as 5 and requires the symmetric
    // u4b8 form (linear.cpp:1418-1435): it is served by the same kernels with sym = 1 (no Marlin repack needed).
    zl_llama_config_t norm_cfg = *cfg;
    if (norm_cfg.quant_type == 8) {
        norm_cfg.quant_type = 5;
        norm_cfg.sym = 1;
    }
    cfg = &norm_cfg;
    ZL_CHECK_SUPPORTED(cfg->quant_type == 0 || cfg->quant_type == 2 || cfg->quant_type == 5 || cfg->quant_type == 6 ||
                       cfg->quant_type == 7);
    ZL_CHECK_SUPPORTED(!(cfg->quant_type == 5 || cfg->quant_type == 6) || cfg->dtype == ZL_F16);
    ZL_CHECK_SUPPORTED(!(cfg->quant_type == 2 || cfg->quant_type == 7) || cfg->tp_size == 1);   // "A must be half" q_gemm_k_major.cu:989
    ZL_CHECK_SUPPORTED(cfg->dtype == ZL_F16 || cfg->dtype == ZL_BF16);
    ZL_CHECK_SUPPORTED(cfg->tp_size >= 1 && cfg->tp_rank >= 0 && cfg->tp_rank < cfg->tp_size);
    ZL_CHECK_SUPPORTED(cfg->num_heads % cfg->tp_size == 0 && cfg->num_kv_heads % cfg->tp_size == 0 &&
                       cfg->dim_ff % cfg->tp_size == 0 && cfg->vocab_size % cfg->tp_size == 0);
    ZL_CHECK_SUPPORTED(!(cfg->quant_type == 5 || cfg->quant_type == 6) || cfg->group_size == zl::kW4GroupK);
    ZL_CHECK_ARG(cfg->fuse >= 0 && cfg->fuse <= 3);
    ZL_CHECK_ARG(cfg->prefill_chunk >= 0 && cfg->prefill_chunk <= 2048);
    ZL_CHECK_SUPPORTED(cfg->fuse < 2 || cfg->dim_head % 32 == 0);
    RCHECK(zl_prepare());
    zl_llama* m = new zl_llama();
    m->cfg = *cfg;
    m->hq = cfg->num_heads / cfg->tp_size;
    m->hkv = cfg->num_kv_heads / cfg->tp_size;
    m->ff = cfg->dim_ff / cfg->tp_size;
    m->vshard = cfg->vocab_size / cfg->tp_size;
    m->layers.resize(cfg->num_layers);
    if (cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete m;
        zl_set_last_error(__FILE__, __LINE__, "cudaStreamCreate failed (no CUDA device? there is no CPU fallback)");
        return ZL_ERR_CUDA;
    }
    *out = m;
    return ZL_OK;
}

extern "C" int zl_llama_set_comm(zl_llama_t* m, zl_comm_t* comm) {
    ZL_CHECK_ARG(m && comm);
    ZL_CHECK_ARG(zl_comm_world_size(comm) == m->cfg.tp_size && zl_comm_rank(comm) == m->cfg.tp_rank);
    m->comm = comm;
    return ZL_OK;
}

extern "C" void zl_llama_destroy(zl_llama_t* m) {
    if (!m) return;
    cudaStreamSynchronize(m->stream);
    for (auto& g : m->graphs) cudaGraphExecDestroy(g.second);
    for (auto& s : m->staged) cudaFree(s.second.ptr);
    for (auto& L : m->layers) {
        for (void* p : {L.ln_attn, L.ln_ff, L.q_qkv.packed, L.q_qkv.bias, L.q_o.packed, L.q_o.bias, L.q_gu.packed,
                        L.q_down.packed, L.q_down.bias, L.q_qkv.packed_i, L.q_o.packed_i, L.q_gu.packed_i, L.q_down.packed_i, L.d_qkv.w, L.d_qkv.bias, L.d_o.w, L.d_o.bias, L.d_gu.w,
                        L.d_gu.bias, L.d_down.w, L.d_down.bias, L.d_qkv.w8, L.d_qkv.w_scale, L.d_o.w8, L.d_o.w_scale, L.d_gu.w8, L.d_gu.w_scale, L.d_down.w8, L.d_down.w_scale, L.kbuf, L.vbuf, (void*)L.k_addrs, (void*)L.v_addrs})
            if (p) cudaFree(p);
    }
    for (void* p : {m->emb, m->lm_head_tied ? nullptr : m->lm_head, m->ln_f, m->h, m->xn, m->qkv, m->q, m->ao, m->act,
                    m->pend, m->gu, (void*)m->logits, (void*)m->cosb, (void*)m->sinb, (void*)m->d_tokens,
                    m->h2, (void*)m->d_pos, (void*)m->d_lens, (void*)m->d_next, (void*)m->d_iota, m->attn_ws, m->argmax_ws, (void*)m->d_tb, (void*)m->d_mask, m->xq, (void*)m->xs,
                    (void*)m->d_sparams, (void*)m->d_seen, (void*)m->d_draws})
        if (p) cudaFree(p);
    if (m->reduce_stream) {
        cudaStreamSynchronize(m->reduce_stream);
        for (int h = 0; h < 2; ++h)
            for (cudaEvent_t e : {m->ev_o[h], m->ev_r1[h], m->ev_dn[h], m->ev_r2[h]})
                if (e) cudaEventDestroy(e);
        cudaStreamDestroy(m->reduce_stream);
    }
    if (m->h_stage) cudaFreeHost(m->h_stage);
    if (m->h_ring) cudaFreeHost(m->h_ring);
    for (cudaEvent_t e : m->ring_ev)
        if (e) cudaEventDestroy(e);
    for (void* p : {(void*)m->d_pf_tokens, (void*)m->d_pf_pos})
        if (p) cudaFree(p);
    cudaStreamDestroy(m->stream);
    delete m;
}

extern "C" int zl_llama_load_tensor(zl_llama_t* m, const char* name, const void* data_host, int rows, int cols,
                                    int elem_bytes) {
    ZL_CHECK_ARG(m && name && data_host && rows > 0 && cols > 0 && elem_bytes > 0);
    if (m->finalized) {
        zl_set_last_error(__FILE__, __LINE__, "model already finalized");
        return ZL_ERR_STATE;
    }
    Staged s;
    s.rows = rows;
    s.cols = cols;
    s.elem = elem_bytes;
    const size_t bytes = (size_t)rows * cols * elem_bytes;
    RCHECK(dmalloc(&s.ptr, bytes));
    ZL_CHECK_CUDA(cudaMemcpyAsync(s.ptr, data_host, bytes, cudaMemcpyHostToDevice, m->stream));
    ZL_CHECK_CUDA(cudaStreamSynchronize(m->stream));
    drop(m, name);
    m->staged[name] = s;
    return ZL_OK;
}

extern "C" int zl_llama_finalize(zl_llama_t* m) {
    ZL_CHECK_ARG(m);
    if (m->finalized) return ZL_OK;
    for (int l = 0; l < m->cfg.num_layers; ++l)
        if (!m->layers[l].ln_attn) RCHECK(finalize_layer(m, l));
    RCHECK(finalize_globals(m));
    RCHECK(alloc_runtime(m));
    m->finalized = true;
    return ZL_OK;
}

namespace {
int stage_random(zl_llama* m, const std::string& name, int rows, int cols, int elem, int kind, float lo, float hi,
                 uint64_t seed) {
    Staged s;
    s.rows = rows;
    s.cols = cols;
    s.elem = elem;
    const size_t n = (size_t)rows * cols;
    RCHECK(dmalloc(&s.ptr, n * elem));
    uint64_t h = seed;
    for (char ch : name) h = h * 1099511628211ull + (unsigned char)ch;
    if (kind == 0)
        RCHECK(zl_fill_random_u32((uint32_t*)s.ptr, n, h, m->stream));
    else if (kind == 1)
        RCHECK(zl_fill_const_u32((uint32_t*)s.ptr, n, 0x77777777u, m->stream));
    else
        RCHECK(zl_fill_uniform(s.ptr, n, lo, hi, h, m->cfg.dtype, m->stream));
    m->staged[name] = s;
    return ZL_OK;
}

int stage_random_linear(zl_llama* m, const std::string& prefix, int K, int N, uint64_t seed) {
    const auto& c = m->cfg;
    if (c.quant_type == 5) {
        const int G = K / c.group_size;
        RCHECK(stage_random(m, prefix + ".qweight", K / 8, N, 4, 0, 0, 0, seed));
        if (c.sym) {
            const size_t words = (size_t)(K / 8) * N;
            k_recentre_nibbles<<<(unsigned)((words + 255) / 256), 256, 0, m->stream>>>(
                static_cast<uint32_t*>(m->staged[prefix + ".qweight"].ptr), words);
            ZL_CHECK_LAUNCH();
        }
        RCHECK(stage_random(m, prefix + ".qzeros", G, N / 8, 4, c.sym ? 1 : 0, 0, 0, seed));
        RCHECK(stage_random(m, prefix + ".scales", G, N, 2, 2, 0.002f, 0.006f, seed));   // SURVEY 8d config 3
    } else if (c.quant_type == 6) {
        const int G = K / c.group_size;
        RCHECK(stage_random(m, prefix + ".qweight", K, N / 8, 4, 0, 0, 0, seed));
        RCHECK(stage_random(m, prefix + ".qzeros", G, N / 8, 4, 0, 0, 0, seed));
        RCHECK(stage_random(m, prefix + ".scales", G, N, 2, 2, 0.002f, 0.006f, seed));
    } else if (c.quant_type == 7) {
        // random e4m3 codes with the exponent MSB cleared (|w| < 2, no NaN encodings) and a per-tensor scale
        RCHECK(stage_random(m, prefix + ".weight", N, K / 4, 4, 0, 0, 0, seed));
        Staged& w = m->staged[prefix + ".weight"];
        const size_t words = (size_t)N * K / 4;
        k_and_u32<<<(unsigned)((words + 255) / 256), 256, 0, m->stream>>>(static_cast<uint32_t*>(w.ptr), words, 0xBFBFBFBFu);
        ZL_CHECK_LAUNCH();
        w.cols = K;
        w.elem = 1;
        Staged sc;
        sc.rows = sc.cols = 1;
        sc.elem = 4;
        RCHECK(dmalloc(&sc.ptr, 4));
        k_set_f32<<<1, 1, 0, m->stream>>>(static_cast<float*>(sc.ptr), 0.03f);
        ZL_CHECK_LAUNCH();
        m->staged[prefix + ".weight_scale"] = sc;
    } else {
        RCHECK(stage_random(m, prefix + ".weight", N, K, 2, 2, -0.035f, 0.035f, seed));   // ~ randn*0.02
    }
    return ZL_OK;
}
}  // namespace

extern "C" int zl_llama_init_synthetic(zl_llama_t* m, uint64_t seed) {
    ZL_CHECK_ARG(m);
    if (m->finalized) {
        zl_set_last_error(__FILE__, __LINE__, "model already finalized");
        return ZL_ERR_STATE;
    }
    const auto& c = m->cfg;
    const int D = c.dim_model, d = c.dim_head;
    for (int l = 0; l < c.num_layers; ++l) {
        const std::string p = "layers." + std::to_string(l) + ".";
        RCHECK(stage_random(m, p + "ln_attn.weight", 1, D, 2, 2, 0.9f, 1.1f, seed));
        RCHECK(stage_random(m, p + "ln_ff.weight", 1, D, 2, 2, 0.9f, 1.1f, seed));
        RCHECK(stage_random_linear(m, p + "attn.project_q", D, m->hq * d, seed));
        RCHECK(stage_random_linear(m, p + "attn.project_k", D, m->hkv * d, seed));
        RCHECK(stage_random_linear(m, p + "attn.project_v", D, m->hkv * d, seed));
        if (c.qkv_bias) {
            RCHECK(stage_random(m, p + "attn.project_q.bias", 1, m->hq * d, 2, 2, -0.03f, 0.03f, seed));
            RCHECK(stage_random(m, p + "attn.project_k.bias", 1, m->hkv * d, 2, 2, -0.03f, 0.03f, seed));
            RCHECK(stage_random(m, p + "attn.project_v.bias", 1, m->hkv * d, 2, 2, -0.03f, 0.03f, seed));
        }
        RCHECK(stage_random_linear(m, p + "attn.attn_out", m->hq * d, D, seed));
        RCHECK(stage_random_linear(m, p + "ff.w_in", D, m->ff, seed));
        RCHECK(stage_random_linear(m, p + "ff.w_gated", D, m->ff, seed));
        RCHECK(stage_random_linear(m, p + "ff.w_out", m->ff, D, seed));
        RCHECK(finalize_layer(m, l));   // bound the staging memory to one layer
    }
    RCHECK(stage_random(m, "token_embedding.weight", c.vocab_size, D, 2, 2, -0.035f, 0.035f, seed));
    RCHECK(stage_random(m, "output_layernorm.weight", 1, D, 2, 2, 0.9f, 1.1f, seed));
    RCHECK(stage_random(m, "lm_head.weight", m->vshard, D, 2, 2, -0.035f, 0.035f, seed + 7919 * c.tp_rank));
    return zl_llama_finalize(m);
}

extern "C" int zl_llama_set_state(zl_llama_t* m, const int32_t* tokens_host, const int32_t* positions_host,
                                  int B) {
    ZL_CHECK_ARG(m && tokens_host && positions_host && B > 0 && B <= m->cfg.max_batch);
    if (!m->finalized) {
        zl_set_last_error(__FILE__, __LINE__, "model not finalized");
        return ZL_ERR_STATE;
    }
    const int slot = m->ring_next;
    m->ring_next = (slot + 1) % zl_llama::kStageSlots;
    if (m->ring_used[slot]) ZL_CHECK_CUDA(cudaEventSynchronize(m->ring_ev[slot]));   // its previous copies have executed
    int32_t* hs = m->h_ring + (size_t)slot * 2 * m->cfg.max_batch;
    int mx = 0;
    for (int i = 0; i < B; ++i) {
        ZL_CHECK_ARG(positions_host[i] >= 0 && positions_host[i] < m->cfg.max_seq);
        ZL_CHECK_ARG(tokens_host[i] >= 0 && tokens_host[i] < m->cfg.vocab_size);
        hs[i] = tokens_host[i];
        hs[B + i] = positions_host[i];
        if (positions_host[i] + 1 > mx) mx = positions_host[i] + 1;
    }
    m->cur_max_len = mx;
    ZL_CHECK_CUDA(cudaMemcpyAsync(m->d_tokens, hs, B * 4, cudaMemcpyHostToDevice, m->stream));
    ZL_CHECK_CUDA(cudaMemcpyAsync(m->d_pos, hs + B, B * 4, cudaMemcpyHostToDevice, m->stream));
    ZL_CHECK_CUDA(cudaEventRecord(m->ring_ev[slot], m->stream));
    m->ring_used[slot] = true;
    return ZL_OK;
}

extern "C" int zl_llama_step_device(zl_llama_t* m, int B) {
    ZL_CHECK_ARG(m && B > 0 && B <= m->cfg.max_batch);
    if (m->cur_max_len >= m->cfg.max_seq) {
        zl_set_last_error(__FILE__, __LINE__, "KV buffers full (max_seq reached)");
        return ZL_ERR_STATE;
    }
    RCHECK(run_step(m, B));
    k_advance<<<cdiv(B, 64), 64, 0, m->stream>>>(m->d_tokens, m->d_pos, m->d_next, B, g_w4_trace);
    ZL_CHECK_LAUNCH();
    m->cur_max_len += 1;
    return ZL_OK;
}

extern "C" int zl_llama_decode(zl_llama_t* m, const int32_t* tokens_host, const int32_t* positions_host, int B,
                               int32_t* next_tokens_host, float* logits_host) {
    ZL_CHECK_ARG(next_tokens_host != nullptr);
    RCHECK(zl_llama_set_state(m, tokens_host, positions_host, B));
    RCHECK(run_step(m, B));
    ZL_CHECK_CUDA(cudaMemcpyAsync(m->h_stage + 3 * B, m->d_next, B * 4, cudaMemcpyDeviceToHost, m->stream));
    if (logits_host)   // (B, vocab/tp) of this rank's shard
        ZL_CHECK_CUDA(cudaMemcpyAsync(logits_host, m->logits, (size_t)B * m->vshard * 4, cudaMemcpyDeviceToHost,
                                      m->stream));
    ZL_CHECK_CUDA(cudaStreamSynchronize(m->stream));
    for (int i = 0; i < B; ++i) next_tokens_host[i] = m->h_stage[3 * B + i];
    return ZL_OK;
}

extern "C" int zl_llama_get_state(zl_llama_t* m, int32_t* tokens_host, int32_t* positions_host, int B) {
    ZL_CHECK_ARG(m && tokens_host && positions_host && B > 0 && B <= m->cfg.max_batch);
    ZL_CHECK_CUDA(cudaMemcpyAsync(m->h_stage, m->d_tokens, B * 4, cudaMemcpyDeviceToHost, m->stream));
    ZL_CHECK_CUDA(cudaMemcpyAsync(m->h_stage + B, m->d_pos, B * 4, cudaMemcpyDeviceToHost, m->stream));
    ZL_CHECK_CUDA(cudaStreamSynchronize(m->stream));
    for (int i = 0; i < B; ++i) {
        tokens_host[i] = m->h_stage[i];
        positions_host[i] = m->h_stage[B + i];
    }
    return ZL_OK;
}

extern "C" int zl_llama_get_logits(zl_llama_t* m, float* logits_host, int B) {
    ZL_CHECK_ARG(m && logits_host && B > 0 && B <= m->cfg.max_batch);
    if (!m->finalized) {
        zl_set_last_error(__FILE__, __LINE__, "model not finalized");
        return ZL_ERR_STATE;
    }
    ZL_CHECK_CUDA(cudaMemcpyAsync(logits_host, m->logits, (size_t)B * m->vshard * 4, cudaMemcpyDeviceToHost, m->stream));
    ZL_CHECK_CUDA(cudaStreamSynchronize(m->stream));
    return ZL_OK;
}

extern "C" int zl_llama_bench_gemms(zl_llama_t* m, int B, int iters, float* ms, int* launches, double* bytes) {
    ZL_CHECK_ARG(m && B > 0 && B <= m->cfg.max_batch && iters > 0 && ms);
    const auto& c = m->cfg;
    const int D = c.dim_model, d = c.dim_head, dt = c.dtype, pdl = c.use_pdl;
    const bool w4 = c.quant_type == 5 || c.quant_type == 6;
    cudaStream_t st = m->stream;
    (void)pdl;
    cudaEvent_t e0, e1;
    ZL_CHECK_CUDA(cudaEventCreate(&e0));
    ZL_CHECK_CUDA(cudaEventCreate(&e1));
    int n_launch = 0;
    double nbytes = 0;
    for (int it = -1; it < iters; ++it) {   // it == -1: warm-up pass
        if (it == 0) ZL_CHECK_CUDA(cudaEventRecord(e0, st));
        for (int l = 0; l < c.num_layers; ++l) {
            Layer& L = m->layers[l];
            if (w4) {
                // the SAME kernel variants as the decode step (enqueue_step): fused RMSNorm prologue, qkv RoPE + KV-append
                // epilogue, SwiGLU, residual epilogues, per-kernel PDL policy.  (Rewrites the KV rows of the current
                // positions and the residual stream: call it after the measurements that need the decode state.)
                const void* ln1 = c.fuse >= 1 ? L.ln_attn : nullptr;
                const void* ln2 = c.fuse >= 1 ? L.ln_ff : nullptr;
                m->cur_tb = m->d_iota;
                m->cur_pos = m->d_pos;
                if (c.fuse >= 2)
                    RCHECK(w4_gemm(m, m->h, D, L.q_qkv, nullptr, nullptr, B, ZL_EPI_QKV_ROPE, ln1, &L, l, 0));
                else
                    RCHECK(w4_gemm(m, ln1 ? m->h : m->xn, D, L.q_qkv, nullptr, m->qkv, B, ZL_EPI_NONE, ln1, nullptr, l, 0));
                RCHECK(w4_gemm(m, m->ao, m->hq * d, L.q_o, m->h, m->h, B, ZL_EPI_RESIDUAL, nullptr, nullptr, l, 2));
                RCHECK(w4_gemm(m, ln2 ? m->h : m->xn, D, L.q_gu, nullptr, m->act, B, ZL_EPI_SWIGLU, ln2, nullptr, l, 3));
                RCHECK(w4_gemm(m, m->act, m->ff, L.q_down, m->h, m->h, B, ZL_EPI_RESIDUAL, nullptr, nullptr, l, 4));
                if (it == 0) {
                    nbytes += (double)zl_w4_packed_bytes(L.q_qkv.N, D, c.group_size) +
                              (double)zl_w4_packed_bytes(D, m->hq * d, c.group_size) +
                              (double)zl_w4_packed_bytes(L.q_gu.N, D, c.group_size) +
                              (double)zl_w4_packed_bytes(D, m->ff, c.group_size);
                    // activations in/out (fp16)
                    nbytes += 2.0 * B * (D + L.q_qkv.N + m->hq * d + 2 * D + D + m->ff + m->ff + 2 * D);
                }
            } else {
                RCHECK(dense_or_w8(m, m->xn, L.d_qkv, m->qkv, B, pdl));
                RCHECK(dense_or_w8(m, m->ao, L.d_o, m->pend, B, pdl));
                RCHECK(dense_or_w8(m, m->xn, L.d_gu, m->gu, B, pdl));
                RCHECK(dense_or_w8(m, m->act, L.d_down, m->pend, B, pdl));
                if (it == 0) {
                    // weight bytes: 2 per element dense, 1 (+ per-row scale) for W8A8 (SURVEY 8d)
                    const double wb = L.d_qkv.w8 ? 1.0 : 2.0;
                    nbytes += wb * ((double)L.d_qkv.N * D + (double)D * m->hq * d + 2.0 * m->ff * D + (double)D * m->ff) +
                              2.0 * B * (D + L.d_qkv.N + m->hq * d + D + D + 2 * m->ff + m->ff + D);
                }
            }
            if (it == 0) n_launch += 4;
        }
    }
    ZL_CHECK_CUDA(cudaEventRecord(e1, st));
    ZL_CHECK_CUDA(cudaEventSynchronize(e1));
    ZL_CHECK_CUDA(cudaEventElapsedTime(ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (launches) *launches = n_launch;
    if (bytes) *bytes = nbytes;
    return ZL_OK;
}

extern "C" int zl_llama_sync(zl_llama_t* m) {
    ZL_CHECK_ARG(m);
    ZL_CHECK_CUDA(cudaStreamSynchronize(m->stream));
    return ZL_OK;
}

extern "C" int zl_llama_prefill(zl_llama_t* m, int task, const int32_t* tokens_host, int n, int pos0,
                                int32_t* next_token_host, float* logits_host) {
    ZL_CHECK_ARG(m && m->finalized && tokens_host && next_token_host && n > 0 && pos0 >= 0);
    ZL_CHECK_ARG(task >= 0 && task < m->cfg.max_batch);
    const int chunk = m->cfg.prefill_chunk;
    if (chunk <= 0) {
        zl_set_last_error(__FILE__, __LINE__, "zl_llama_prefill needs cfg.prefill_chunk > 0");
        return ZL_ERR_STATE;
    }
    if (pos0 + n > m->cfg.max_seq) {
        zl_set_last_error(__FILE__, __LINE__, "prompt does not fit the KV buffers (max_seq)");
        return ZL_ERR_STATE;
    }
    int32_t* h_tok = m->h_stage + 4 * m->cfg.max_batch + 4;   // pinned staging for one chunk of token ids
    for (int c0 = 0; c0 < n; c0 += chunk) {
        const int cn = (n - c0) < chunk ? (n - c0) : chunk;
        if (c0 > 0) ZL_CHECK_CUDA(cudaStreamSynchronize(m->stream));   // staging buffer reuse
        for (int i = 0; i < cn; ++i) {
            ZL_CHECK_ARG(tokens_host[c0 + i] >= 0 && tokens_host[c0 + i] < m->cfg.vocab_size);
            h_tok[i] = tokens_host[c0 + i];
        }
        ZL_CHECK_CUDA(cudaMemcpyAsync(m->d_pf_tokens, h_tok, cn * 4, cudaMemcpyHostToDevice, m->stream));
        PrefillChunk pc{task, pos0 + c0, cn, c0 + cn == n};
        RCHECK(enqueue_step(m, 1, 0, &pc));
    }
    ZL_CHECK_CUDA(cudaMemcpyAsync(m->h_stage + 3 * m->cfg.max_batch, m->d_next, 4, cudaMemcpyDeviceToHost, m->stream));
    if (logits_host)
        ZL_CHECK_CUDA(cudaMemcpyAsync(logits_host, m->logits, (size_t)m->vshard * 4, cudaMemcpyDeviceToHost, m->stream));
    ZL_CHECK_CUDA(cudaStreamSynchronize(m->stream));
    *next_token_host = m->h_stage[3 * m->cfg.max_batch];
    if (pos0 + n > m->cur_max_len) m->cur_max_len = pos0 + n;
    return ZL_OK;
}

extern "C" int zl_llama_set_sampling(zl_llama_t* m, int task, const zl_sample_params_t* host_params) {
    ZL_CHECK_ARG(m && host_params);
    if (m->cfg.tp_size > 1) {
        zl_set_last_error(__FILE__, __LINE__,
                          "unsupported: sampling with tp_size > 1 (top-p over vocabulary shards needs a global select)");
        return ZL_ERR_UNSUPPORTED;
    }
    if (!m->finalized) {
        zl_set_last_error(__FILE__, __LINE__, "model not finalized");
        return ZL_ERR_STATE;
    }
    ZL_CHECK_ARG(task >= 0 && task < m->cfg.max_batch);
    const zl_sample_params_t& p = *host_params;
    // random_util.cu:121-122
    ZL_CHECK_ARG(p.temperature > 0.0f && p.temperature <= 3.0e38f);
    ZL_CHECK_ARG(p.top_p >= 0.0f && p.top_p <= 1.0f);
    ZL_CHECK_ARG(p.top_k >= 0 && p.top_k < m->cfg.vocab_size);
    ZL_CHECK_ARG(p.repetition_penalty > 0.0f && p.repetition_penalty <= 3.0e38f);
    ZL_CHECK_ARG(p.presence_penalty == p.presence_penalty && p.presence_penalty >= -3.0e38f &&
                 p.presence_penalty <= 3.0e38f);
    RCHECK(write_sampling(m, task, p));
    m->sampling[task] = 1;
    return ZL_OK;
}

extern "C" int zl_llama_clear_sampling(zl_llama_t* m, int task) {
    ZL_CHECK_ARG(m);
    if (!m->finalized) {
        zl_set_last_error(__FILE__, __LINE__, "model not finalized");
        return ZL_ERR_STATE;
    }
    ZL_CHECK_ARG(task >= 0 && task < m->cfg.max_batch);
    if (m->cfg.tp_size > 1) return ZL_OK;   // never set
    RCHECK(write_sampling(m, task, kGreedyParams));
    m->sampling[task] = 0;
    return ZL_OK;
}

extern "C" zl_stream_t zl_llama_stream(zl_llama_t* m) { return m ? (zl_stream_t)m->stream : nullptr; }

extern "C" int zl_llama_stats(zl_llama_t* m, int B, double* weight_bytes, int* kernels_per_step) {
    ZL_CHECK_ARG(m);
    (void)B;
    if (weight_bytes) *weight_bytes = m->weight_bytes;
    if (kernels_per_step) *kernels_per_step = m->kernels_per_step;
    return ZL_OK;
}
