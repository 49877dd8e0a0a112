// Batch decode attention over per-task ragged KV buffers (GQA/MQA), split-KV with LSE combine.
//
// Replaces nn::multi_query_attention_rag_buffer and its kernels KERNEL_mqa_rag_buffer1 /
// KERNEL_mqa_rag_buffer_split_kv / KERNEL_mqa_combine / the wmma KERNEL_mqa_rag_buffer
// (reference src/nn/attention/attention_kernel.cu:674-725, 730-923, 926-1017, 1252-1457).
//
// One CTA = (kv-split, kv-head, task x query).  The whole GQA group (<= 8 q-heads per pass) shares
// every K/V byte: K is read ONCE per kv-head straight into tensor-core A fragments (16 keys x 16 dims),
// Q is the B operand (16 dims x 8 heads), so S = K.Q^T needs no shuffles; softmax is the reference's
// exact two-pass fp32 form inside the split (mask ? scale*s : -inf, max seeded -1e20, sum seeded 1e-20);
// P.V runs in fp32 on the CUDA cores with 16-byte coalesced V loads (each V element feeds all heads).
// Splits are merged with the reference's LSE rule (attention_kernel.cu:881-923).
#include "common.cuh"
#include "decode_attn_short.cuh"
#include "decode_attn_warp.cuh"

#include <cstdlib>
#include <type_traits>

namespace zl {

constexpr int kAttnThreads = 128;
constexpr int kAttnWarps = 4;
constexpr int kAttnMaxRange = 1024;            // keys per CTA; logits live in shared memory
constexpr int kAttnRowStride = kAttnMaxRange + 4;
constexpr int kAttnMaxSplits = 64;
// kernel ids reported by zl_decode_attention_plan
constexpr int kAttnKernelTc = 0;               // k_decode_attn, P.V on the tensor cores
constexpr int kAttnKernelWarp = 1;             // k_decode_attn_warp
constexpr int kAttnKernelShort = 2;            // k_decode_attn_short (ZL_ATTN_OLD_SHORT)
constexpr int kAttnKernelPvFp32 = 3;           // k_decode_attn, P.V on the CUDA cores (ZL_ATTN_PV_FP32)

template <typename T, int D, bool PV_FP32>
__global__ void __launch_bounds__(kAttnThreads)
k_decode_attn(const T* __restrict__ q, const int32_t* __restrict__ buf_lens, T* const* __restrict__ k_addrs,
              T* const* __restrict__ v_addrs, const int8_t* __restrict__ mask, float scale,
              T* __restrict__ out, float* __restrict__ part_o, float* __restrict__ part_m,
              float* __restrict__ part_l, int len_q, int num_heads, int num_kv_heads, int m_query,
              int num_splits, int bshd, const uint8_t* __restrict__ pf_ptr, unsigned long long pf_bytes) {
    constexpr int NI = D / 32;                 // 16-byte chunks per lane per key row
    constexpr int DC = D / 8;                  // threads covering one V row
    constexpr int NSUB = kAttnThreads / DC;    // key subsets in the PV phase
    __shared__ __align__(16) float s_logit[8 * kAttnRowStride];
    __shared__ float s_m[8], s_l[8];

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const int hgroups = (m_query + 7) / 8;
    const int split = blockIdx.x;
    const int hk = blockIdx.y / hgroups, hg = blockIdx.y % hgroups;
    const int bq = blockIdx.z, b = bq / len_q, qi = bq % len_q;
    const int mq0 = hg * 8;
    const int mq = min(8, m_query - mq0);
    const int head0 = hk * m_query + mq0;

    pdl_trigger();
    // attention barely touches HBM at small batch: use the time to pull a later GEMM's weights into L2
    if (pf_ptr) {
        const int n_cta = gridDim.x * gridDim.y * gridDim.z;
        const int cta = blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z);
        const int wpc = blockDim.x >> 5;
        l2_prefetch_lines(pf_ptr, (size_t)pf_bytes, cta * wpc + warp, n_cta * wpc, lane);
    }
    pdl_wait();

    const int len_buf = buf_lens[b];
    const int chunk = attn_round16((len_buf + num_splits - 1) / num_splits);
    const int k0 = split * chunk;
    const int k1 = min(len_buf, k0 + chunk);
    const int n = max(0, k1 - k0);

    const size_t stride = bshd ? (size_t)num_kv_heads * D : (size_t)D;
    const size_t base = bshd ? (size_t)hk * D : (size_t)hk * len_buf * D;
    const T* kbase = k_addrs[b] + base;
    const T* vbase = v_addrs[b] + base;

    const int8_t* mrow = nullptr;
    if (mask) {
        size_t len_off = 0;
        for (int j = 0; j < b; ++j) len_off += buf_lens[j];
        mrow = mask + (size_t)len_q * len_off + (size_t)qi * len_buf;
    }

    // ---- phase 1: S = K.Q^T on tensor cores ----
    uint4 qf[NI];
#pragma unroll
    for (int i = 0; i < NI; ++i) {
        qf[i] = (g < mq) ? ld_cg_u4(q + ((size_t)bq * num_heads + head0 + g) * D + i * 32 + t * 8)
                         : make_uint4(0, 0, 0, 0);
    }
    const int ntiles = (n + 15) >> 4;
    for (int tile = warp; tile < ntiles; tile += kAttnWarps) {
        const int ka_i = k0 + tile * 16 + g, kb_i = ka_i + 8;
        const T* pa = kbase + (size_t)min(ka_i, k1 - 1) * stride + t * 8;
        const T* pb = kbase + (size_t)min(kb_i, k1 - 1) * stride + t * 8;
        uint4 ka[NI], kb[NI];
#pragma unroll
        for (int i = 0; i < NI; ++i) {
            ka[i] = ld_cg_u4(pa + i * 32);
            kb[i] = ld_cg_u4(pb + i * 32);
        }
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int i = 0; i < NI; ++i) {
            const uint32_t a0[4] = {ka[i].x, kb[i].x, ka[i].y, kb[i].y};
            const uint32_t a1[4] = {ka[i].z, kb[i].z, ka[i].w, kb[i].w};
            mma_attn<T>(acc, a0, qf[i].x, qf[i].y);
            mma_attn<T>(acc, a1, qf[i].z, qf[i].w);
        }
        const bool va = ka_i < k1 && (!mrow || mrow[ka_i] != 0);
        const bool vb = kb_i < k1 && (!mrow || mrow[kb_i] != 0);
        const int la = tile * 16 + g;
        const float ninf = -INFINITY;
        if (2 * t < mq) {
            s_logit[(2 * t) * kAttnRowStride + la] = va ? acc[0] * scale : ninf;
            s_logit[(2 * t) * kAttnRowStride + la + 8] = vb ? acc[2] * scale : ninf;
        }
        if (2 * t + 1 < mq) {
            s_logit[(2 * t + 1) * kAttnRowStride + la] = va ? acc[1] * scale : ninf;
            s_logit[(2 * t + 1) * kAttnRowStride + la + 8] = vb ? acc[3] * scale : ninf;
        }
    }
    __syncthreads();

    // ---- phase 2: masked softmax statistics per head (attention_kernel.cu:434-489) ----
    for (int h = warp; h < mq; h += kAttnWarps) {
        float* row = s_logit + h * kAttnRowStride;
        float mx = -1e20f;
        for (int i = lane; i < n; i += 32) mx = fmaxf(mx, row[i]);
        mx = warp_max(mx);
        float sum = 0.f;
        for (int i = lane; i < n; i += 32) {
            const float e = expf(row[i] - mx);
            row[i] = e;
            sum += e;
        }
        sum = warp_sum(sum) + 1e-20f;
        if (lane == 0) {
            s_m[h] = mx;
            s_l[h] = sum;
        }
    }
    __syncthreads();

    // ---- phase 3: O = P.V on the tensor cores (mma.sync m16n8k16, fp32 accumulate); ZL_ATTN_PV_FP32=1 keeps the CUDA-core
    // loop of round 1 (every V element times every head in fp32) for A/B measurements ----
    // A = P [head (8 of 16 rows) x 16 keys]: fp16 models carry p * 2^10 in fp16 (11 significant bits, no subnormals); bf16
    // models carry p as bf16 hi + lo (two MMAs), so that the product keeps ~16 bits of p.  B = V [16 keys x 8 columns]: a B
    // register holds TWO KEYS of one column while V is key-major, so lane (g, t) loads D/8 contiguous elements (columns
    // NJ g ..) of its four keys 2t, 2t+1, 2t+8, 2t+9 and interleaves row pairs with PRMT; n-tile j column c stands for column
    // d = NJ c + j of V (a permutation of the columns, undone when the accumulators are written out).
    constexpr int NJ = D / 8;                 // n-tiles = V columns per lane and key row
    constexpr int NW = NJ / 2;                // 32-bit words of a lane's column chunk (2 elements each)
    constexpr bool kHalf = sizeof(T) == 2 && std::is_same<T, __half>::value;
    float* s_red = s_logit;                   // [warp][h][D], valid after the barrier below
    if constexpr (!PV_FP32) {
        float o[NJ][4];
#pragma unroll
        for (int j = 0; j < NJ; ++j) o[j][0] = o[j][1] = o[j][2] = o[j][3] = 0.f;
        for (int tile = warp; tile < ntiles; tile += kAttnWarps) {
            const int kb = tile * 16;
            uint32_t vw[4][NW];
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int kk = kb + 2 * t + (r & 1) + (r >> 1) * 8;
#pragma unroll
                for (int w = 0; w < NW; ++w) vw[r][w] = 0u;
                if (kk < n) {
                    const T* src = vbase + (size_t)(k0 + kk) * stride + g * NJ;
#pragma unroll
                    for (int w4 = 0; w4 < NW / 4; ++w4) {
                        const uint4 v = ld_cg_u4(src + w4 * 8);
                        vw[r][w4 * 4 + 0] = v.x, vw[r][w4 * 4 + 1] = v.y, vw[r][w4 * 4 + 2] = v.z, vw[r][w4 * 4 + 3] = v.w;
                    }
                }
            }
            uint32_t af[4] = {0u, 0u, 0u, 0u}, al[4] = {0u, 0u, 0u, 0u};
            if (g < mq) {
                const float* pr = s_logit + g * kAttnRowStride + kb + 2 * t;
                const float2 p0 = *reinterpret_cast<const float2*>(pr), p1 = *reinterpret_cast<const float2*>(pr + 8);
                const float q0 = kb + 2 * t < n ? p0.x : 0.f, q1 = kb + 2 * t + 1 < n ? p0.y : 0.f;
                const float q2 = kb + 2 * t + 8 < n ? p1.x : 0.f, q3 = kb + 2 * t + 9 < n ? p1.y : 0.f;
                if constexpr (kHalf) {
                    const __half2 h0 = __floats2half2_rn(q0 * 1024.f, q1 * 1024.f), h1 = __floats2half2_rn(q2 * 1024.f, q3 * 1024.f);
                    af[0] = *reinterpret_cast<const uint32_t*>(&h0);
                    af[2] = *reinterpret_cast<const uint32_t*>(&h1);
                } else {
                    const __nv_bfloat162 h0 = __floats2bfloat162_rn(q0, q1), h1 = __floats2bfloat162_rn(q2, q3);
                    const float2 f0 = __bfloat1622float2(h0), f1 = __bfloat1622float2(h1);
                    const __nv_bfloat162 l0 = __floats2bfloat162_rn(q0 - f0.x, q1 - f0.y), l1 = __floats2bfloat162_rn(q2 - f1.x, q3 - f1.y);
                    af[0] = *reinterpret_cast<const uint32_t*>(&h0);
                    af[2] = *reinterpret_cast<const uint32_t*>(&h1);
                    al[0] = *reinterpret_cast<const uint32_t*>(&l0);
                    al[2] = *reinterpret_cast<const uint32_t*>(&l1);
                }
            }
#pragma unroll
            for (int w = 0; w < NW; ++w) {
#pragma unroll
                for (int e = 0; e < 2; ++e) {            // element 2 w + e of the chunk = n-tile j
                    const uint32_t sel = e ? 0x7632u : 0x5410u;
                    const uint32_t b0 = __byte_perm(vw[0][w], vw[1][w], sel), b1 = __byte_perm(vw[2][w], vw[3][w], sel);
                    mma_attn<T>(o[2 * w + e], af, b0, b1);
                    if constexpr (!kHalf) mma_attn<T>(o[2 * w + e], al, b0, b1);
                }
            }
        }
        __syncthreads();   // everyone is done reading probabilities; reuse s_logit as the reduction buffer
        if (g < mq) {
            const float sc = kHalf ? (1.f / 1024.f) : 1.f;
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                s_red[(warp * 8 + g) * D + NJ * (2 * t) + j] = o[j][0] * sc;
                s_red[(warp * 8 + g) * D + NJ * (2 * t + 1) + j] = o[j][1] * sc;
            }
        }
    } else {
        const int dc = tid % DC, sub = tid / DC;
        float o[8][8];
#pragma unroll
        for (int h = 0; h < 8; ++h)
#pragma unroll
            for (int i = 0; i < 8; ++i) o[h][i] = 0.f;
        const T* vp = vbase + (size_t)k0 * stride + dc * 8;
        constexpr int U = 4;
        for (int key = sub; key < n; key += NSUB * U) {
            uint4 vv[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int kk = key + u * NSUB;
                if (kk < n) vv[u] = ld_cg_u4(vp + (size_t)kk * stride);
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int kk = key + u * NSUB;
                if (kk < n) {
                    float vf[8];
                    unpack8<T>(vv[u], vf);
#pragma unroll
                    for (int h = 0; h < 8; ++h) {
                        if (h < mq) {
                            const float p = s_logit[h * kAttnRowStride + kk];
#pragma unroll
                            for (int i = 0; i < 8; ++i) o[h][i] = fmaf(p, vf[i], o[h][i]);
                        }
                    }
                }
            }
        }
        // reduce key subsets: inside the warp first (lanes with equal dc), then across warps via smem
#pragma unroll
        for (int h = 0; h < 8; ++h)
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                float v = o[h][i];
#pragma unroll
                for (int off = DC; off < 32; off <<= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
                o[h][i] = v;
            }
        __syncthreads();   // everyone is done reading probabilities; reuse s_logit as the reduction buffer
        if (lane < DC) {
#pragma unroll
            for (int h = 0; h < 8; ++h)
                if (h < mq) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) s_red[(warp * 8 + h) * D + lane * 8 + i] = o[h][i];
                }
        }
    }
    __syncthreads();
    for (int e = tid; e < mq * D; e += kAttnThreads) {
        const int h = e / D, d = e % D;
        float v = 0.f;
#pragma unroll
        for (int w = 0; w < kAttnWarps; ++w) v += s_red[(w * 8 + h) * D + d];
        v = v / s_l[h];
        const size_t vh = (size_t)bq * num_heads + head0 + h;
        if (num_splits == 1) {
            out[vh * D + d] = from_f32<T>(v);
        } else {
            part_o[(vh * num_splits + split) * D + d] = v;
            if (d == 0) {
                part_m[vh * num_splits + split] = s_m[h];
                part_l[vh * num_splits + split] = s_l[h];
            }
        }
    }
}


// ---------------------------------------------------------------------------------------------------------
// Latency-optimised variant for the small-batch / short-context regime (B200: 148 SMs, a B=1 decode step has
// 8 kv-heads of work): 512 threads, at most 256 keys per CTA, and EVERY global load of the CTA (q, its K tile,
// its V rows) is issued before the first dependent instruction, so the whole CTA costs one memory round trip
// instead of one per loop iteration.  Same math and split/combine contract as k_decode_attn.
// ---------------------------------------------------------------------------------------------------------
template <typename T, int D>
__global__ void __launch_bounds__(kShortThreads)
k_decode_attn_short(const T* __restrict__ q, const int32_t* __restrict__ buf_lens, T* const* __restrict__ k_addrs,
                    T* const* __restrict__ v_addrs, const int8_t* __restrict__ mask, float scale,
                    T* __restrict__ out, float* __restrict__ part_o, float* __restrict__ part_m,
                    float* __restrict__ part_l, int len_q, int num_heads, int num_kv_heads, int m_query,
                    int num_splits, int bshd, const uint8_t* __restrict__ pf_ptr, unsigned long long pf_bytes) {
    extern __shared__ __align__(16) float s_dyn[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    pdl_trigger();
    // attention barely touches HBM at small batch: use the time to pull a later GEMM's weights into L2
    if (pf_ptr) {
        const int n_cta = gridDim.x * gridDim.y * gridDim.z;
        const int cta = blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z);
        const int wpc = blockDim.x >> 5;
        l2_prefetch_lines(pf_ptr, (size_t)pf_bytes, cta * wpc + warp, n_cta * wpc, lane);
    }
    pdl_wait();
    attn_short_item<T, D>(q, buf_lens, k_addrs, v_addrs, mask, scale, out, part_o, part_m, part_l, len_q, num_heads,
                          num_kv_heads, m_query, num_splits, bshd, (int)blockIdx.x, (int)blockIdx.y, (int)blockIdx.z,
                          s_dyn);
}


// grid (B*len_q*num_heads), block D
template <typename T>
__global__ void k_attn_combine(const float* __restrict__ part_o, const float* __restrict__ part_m,
                               const float* __restrict__ part_l, T* __restrict__ out, int num_splits) {
    const int vh = blockIdx.x, D = blockDim.x, d = threadIdx.x;
    pdl_trigger();
    pdl_wait();
    const float* pm = part_m + (size_t)vh * num_splits;
    const float* pl = part_l + (size_t)vh * num_splits;
    float gm = -1e20f;
    for (int i = 0; i < num_splits; ++i) gm = fmaxf(gm, pm[i]);
    float gs = 0.f;
    for (int i = 0; i < num_splits; ++i) gs += pl[i] * expf(pm[i] - gm);
    float res = 0.f;
    for (int i = 0; i < num_splits; ++i) {
        const float w = pl[i] / gs * expf(pm[i] - gm);
        res += part_o[((size_t)vh * num_splits + i) * D + d] * w;
    }
    out[(size_t)vh * D + d] = from_f32<T>(res);
}

static int attn_num_splits(int B, int len_q, int num_kv_heads, int m_query, int max_len_buf) {
    const int hgroups = (m_query + 7) / 8;
    const int base = B * len_q * num_kv_heads * hgroups;
    const int min_splits = cdiv(max_len_buf, kAttnMaxRange);
    const int want = cdiv(2 * 148, base);
    const int max_useful = cdiv(max_len_buf, 256) > 0 ? cdiv(max_len_buf, 256) : 1;   // >= 256 keys per split
    int s = want < max_useful ? want : max_useful;
    if (s > kAttnMaxSplits) s = kAttnMaxSplits;
    if (s < min_splits) s = min_splits;
    if (s < 1) s = 1;
    return s;
}

}  // namespace zl

using namespace zl;

// one-shot prefetch hint consumed by the next zl_decode_attention call on this thread (set by the decode driver)
static thread_local const uint8_t* g_attn_pf_ptr = nullptr;
static thread_local unsigned long long g_attn_pf_bytes = 0;
extern "C" int zl_decode_attention_set_prefetch(const void* ptr, size_t bytes) {
    g_attn_pf_ptr = static_cast<const uint8_t*>(ptr);
    g_attn_pf_bytes = bytes;
    return ZL_OK;
}

extern "C" size_t zl_decode_attention_workspace_bytes(int B, int len_q, int num_heads, int dim_head,
                                                      int max_len_buf) {
    if (B <= 0 || len_q <= 0 || num_heads <= 0 || dim_head <= 0) return 0;
    int splits = cdiv(max_len_buf > 0 ? max_len_buf : 1, kAttnMaxRange);
    if (splits < kAttnMaxSplits) splits = kAttnMaxSplits;
    return (size_t)B * len_q * num_heads * splits * (dim_head + 2) * sizeof(float);
}

extern "C" int zl_decode_attention_plan(int B, int len_q, int num_heads, int num_kv_heads, int max_len_buf, int* kernel,
                                        int* splits) {
    ZL_CHECK_ARG(kernel && splits && B > 0 && len_q > 0 && max_len_buf > 0);
    ZL_CHECK_ARG(num_heads > 0 && num_kv_heads > 0 && num_heads % num_kv_heads == 0);
    const int m_query = num_heads / num_kv_heads;
    // latency regime: few CTAs of work -> 256-key CTAs that issue all their loads up front
    const int hgroups = (m_query + 7) / 8;
    const int short_splits = cdiv(max_len_buf, kShortRange);
    const bool use_short = short_splits <= kAttnMaxSplits &&
                           (long long)B * len_q * num_kv_heads * hgroups * short_splits <= 4 * 148;
    // default for the latency regime: the warp-per-32-keys kernel (one __syncthreads per CTA); ZL_ATTN_OLD_SHORT=1 keeps the
    // previous 512-thread short kernel and ZL_ATTN_PV_FP32=1 the CUDA-core P.V loop of k_decode_attn, for A/B measurements
    static const bool old_short = getenv("ZL_ATTN_OLD_SHORT") != nullptr;
    static const bool pv_fp32 = getenv("ZL_ATTN_PV_FP32") != nullptr;
    if (use_short) {
        *kernel = old_short ? kAttnKernelShort : kAttnKernelWarp;
        *splits = short_splits;
    } else {
        *kernel = pv_fp32 ? kAttnKernelPvFp32 : kAttnKernelTc;
        *splits = attn_num_splits(B, len_q, num_kv_heads, m_query, max_len_buf);
    }
    return ZL_OK;
}

extern "C" int zl_decode_attention(const void* q, const int32_t* buf_lens, void* const* k_addrs,
                                   void* const* v_addrs, const int8_t* mask, float scale, int max_len_buf,
                                   void* out, int B, int len_q, int num_heads, int num_kv_heads, int dim_head,
                                   int bshd, void* workspace, size_t workspace_bytes, int dtype, int pdl,
                                   zl_stream_t stream) {
    ZL_CHECK_ARG(q && buf_lens && k_addrs && v_addrs && out && B > 0 && len_q > 0 && max_len_buf > 0);
    ZL_CHECK_ARG(num_heads > 0 && num_kv_heads > 0 && num_heads % num_kv_heads == 0);
    ZL_CHECK_SUPPORTED(dim_head == 64 || dim_head == 128);
    ZL_CHECK_SUPPORTED(dtype == ZL_F16 || dtype == ZL_BF16);
    const int m_query = num_heads / num_kv_heads;
    int kernel = 0, splits = 0;
    const int rc = zl_decode_attention_plan(B, len_q, num_heads, num_kv_heads, max_len_buf, &kernel, &splits);
    if (rc != ZL_OK) return rc;
    const size_t vheads = (size_t)B * len_q * num_heads;
    float* part_o = nullptr;
    float* part_m = nullptr;
    float* part_l = nullptr;
    if (splits > 1) {
        const size_t need = vheads * splits * (dim_head + 2) * sizeof(float);
        ZL_CHECK_ARG(workspace != nullptr && workspace_bytes >= need);
        part_o = static_cast<float*>(workspace);
        part_m = part_o + vheads * splits * dim_head;
        part_l = part_m + vheads * splits;
    }
    const int hgroups = (m_query + 7) / 8;
    dim3 grid(splits, num_kv_heads * hgroups, B * len_q), block(kAttnThreads);
#define ZL_ATTN_LAUNCH(TT, DD)                                                                                  \
    if (kernel == kAttnKernelWarp) {                                                                            \
        ZL_CHECK_CUDA(launch(k_decode_attn_warp<TT, DD>, grid, dim3(kWarpAttnWarps * 32),                       \
                             (size_t)warp_attn_smem_floats<DD>() * sizeof(float), stream, pdl != 0, (const TT*)q, \
                             buf_lens, (TT* const*)k_addrs, (TT* const*)v_addrs, mask, scale, (TT*)out, part_o, \
                             part_m, part_l, len_q, num_heads, num_kv_heads, m_query, splits, bshd));            \
    } else if (kernel == kAttnKernelShort) {                                                                    \
        static bool attr_set = false;                                                                           \
        if (!attr_set) {                                                                                        \
            ZL_CHECK_CUDA(cudaFuncSetAttribute(k_decode_attn_short<TT, DD>,                                     \
                                               cudaFuncAttributeMaxDynamicSharedMemorySize,                     \
                                               short_smem_bytes<DD>()));                                        \
            attr_set = true;                                                                                    \
        }                                                                                                       \
        ZL_CHECK_CUDA(launch(k_decode_attn_short<TT, DD>, grid, dim3(kShortThreads), short_smem_bytes<DD>(),    \
                             stream, pdl != 0, (const TT*)q, buf_lens, (TT* const*)k_addrs,                     \
                             (TT* const*)v_addrs, mask, scale, (TT*)out, part_o, part_m, part_l, len_q,         \
                             num_heads, num_kv_heads, m_query, splits, bshd, g_attn_pf_ptr, g_attn_pf_bytes));                                  \
    } else                                                                                                      \
    if (kernel == kAttnKernelPvFp32) {                                                                          \
        ZL_CHECK_CUDA(launch(k_decode_attn<TT, DD, true>, grid, block, 0, stream, pdl != 0, (const TT*)q, buf_lens, \
                             (TT* const*)k_addrs, (TT* const*)v_addrs, mask, scale, (TT*)out, part_o, part_m,   \
                             part_l, len_q, num_heads, num_kv_heads, m_query, splits, bshd, g_attn_pf_ptr,      \
                             g_attn_pf_bytes));                                                                 \
    } else                                                                                                      \
    ZL_CHECK_CUDA(launch(k_decode_attn<TT, DD, false>, grid, block, 0, stream, pdl != 0, (const TT*)q, buf_lens, \
                         (TT* const*)k_addrs, (TT* const*)v_addrs, mask, scale, (TT*)out, part_o, part_m,       \
                         part_l, len_q, num_heads, num_kv_heads, m_query, splits, bshd, g_attn_pf_ptr, g_attn_pf_bytes)); \
    if (splits > 1)                                                                                             \
        ZL_CHECK_CUDA(launch(k_attn_combine<TT>, dim3((unsigned)vheads), dim3(DD), 0, stream, pdl != 0,         \
                             (const float*)part_o, (const float*)part_m, (const float*)part_l, (TT*)out, splits));
    if (dtype == ZL_F16) {
        if (dim_head == 128) { ZL_ATTN_LAUNCH(__half, 128) } else { ZL_ATTN_LAUNCH(__half, 64) }
    } else {
        if (dim_head == 128) { ZL_ATTN_LAUNCH(__nv_bfloat16, 128) } else { ZL_ATTN_LAUNCH(__nv_bfloat16, 64) }
    }
#undef ZL_ATTN_LAUNCH
    g_attn_pf_ptr = nullptr;
    g_attn_pf_bytes = 0;
    return ZL_OK;
}
