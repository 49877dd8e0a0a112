// Decode attention over an int8 KV cache (KV_CACHE_DTYPE=int8 of the reference) and the quantising KV append.
//
// Replaces KERNEL_mqa_rag_buffer_split_kv_quant + DEV_mul_qk_quant_h128 / DEV_mul_logit_scale / DEV_mul_score_v_v1
// (reference src/nn/attention/attention_kernel.cu:804-880, src/nn/attention/quant_attention.cuh:10-123) and the
// cache-side quantisation int8_op::quant_calc_scale(x, 127, 128) + copy_to_rag_buffer2 of Attention::attn_search_rag
// (src/nn/attention/attention.cpp:656-676, src/nn/quant/int8/quant_kernel.cu:15-47).
//
// Cache contract (BSHD): per task K / V buffers (len_buf, H_kv, d) uint8 = round(x * 127 / absmax) + 128 and
// scale buffers (len_buf, H_kv) fp32 = absmax / 127, one scale per (token, kv head).  q is fp16.
//   logit[key] = scale * scale_k[key] * sum_d q[d] * (k[key, d] - 128)         (mask ? ... : -inf)
//   out[d]     = sum_key softmax(logit)[key] * scale_v[key] * (v[key, d] - 128)
// Same CTA decomposition as k_decode_attn (decode_attn.cu): one CTA per (kv split, kv head group, task x query), the whole
// GQA group shares every cache byte; K bytes become exact fp16 integers (PRMT 0x64xx magic) and feed mma.sync with fp32
// accumulation -- the reference multiplies and pair-adds in fp16 (quant_attention.cuh:60-70), so ours is the closer one
// to the exact result.  Half the algorithmic bytes of the fp16 cache: 2 * H_kv * d * ctx + 8 * H_kv * ctx per task per layer.
#include "common.cuh"
#include "decode_attn_short.cuh"

namespace zl {

constexpr int kA8Threads = 128;
constexpr int kA8Warps = 4;
constexpr int kA8MaxRange = 1024;
constexpr int kA8RowStride = kA8MaxRange + 4;
constexpr int kA8MaxSplits = 64;

// 4 cache bytes -> 4 exact fp16 integers (u8 - 128): 0x64xx = 1024 + x, minus 1152
__device__ __forceinline__ void u8x4_to_h2x2(uint32_t b, uint32_t& h01, uint32_t& h23) {
    uint32_t a0 = __byte_perm(b, 0x64646464u, 0x4140), a1 = __byte_perm(b, 0x64646464u, 0x4342);
    const __half2 off = __float2half2_rn(1152.f);
    __half2 r0 = __hsub2(*reinterpret_cast<__half2*>(&a0), off), r1 = __hsub2(*reinterpret_cast<__half2*>(&a1), off);
    h01 = *reinterpret_cast<uint32_t*>(&r0);
    h23 = *reinterpret_cast<uint32_t*>(&r1);
}
// one cache byte -> float(u8) - 128 via the 2^23 magic
__device__ __forceinline__ float u8_to_f32(uint32_t word, int i) {
    const uint32_t sel = 0x7540u | (uint32_t)i;
    return __uint_as_float(__byte_perm(word, 0x4B000000u, sel)) - 8388736.f;
}
__device__ __forceinline__ uint2 ld_cg_b8(const void* p) {
    uint2 r;
    asm volatile("ld.global.cg.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}

template <typename TO, int D>
__global__ void __launch_bounds__(kA8Threads)
k_decode_attn_kv8(const __half* __restrict__ q, const int32_t* __restrict__ buf_lens, uint8_t* const* __restrict__ k_addrs,
                  uint8_t* const* __restrict__ v_addrs, float* const* __restrict__ sk_addrs,
                  float* const* __restrict__ sv_addrs, const int8_t* __restrict__ mask, float scale, TO* __restrict__ out,
                  float* __restrict__ part_o, float* __restrict__ part_m, float* __restrict__ part_l, int len_q,
                  int num_heads, int num_kv_heads, int m_query, int num_splits) {
    constexpr int NI = D / 32;                 // 8-byte chunks per lane per key row
    constexpr int DC = D / 8;                  // threads covering one V row (8 bytes each)
    constexpr int NSUB = kA8Threads / DC;
    __shared__ __align__(16) float s_logit[8 * kA8RowStride];
    __shared__ float s_m[8], s_l[8];
    __shared__ int s_wexp;                     // binary exponent of the largest V scale of the CTA's keys

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
    pdl_wait();

    const int len_buf = buf_lens[b];
    const int chunk = attn_round16((len_buf + num_splits - 1) / num_splits);
    const int k0 = split * chunk;
    const int k1 = min(len_buf, k0 + chunk);
    const int n = max(0, k1 - k0);

    const size_t stride = (size_t)num_kv_heads * D;          // BSHD, bytes
    const uint8_t* kbase = k_addrs[b] + (size_t)hk * D;
    const uint8_t* vbase = v_addrs[b] + (size_t)hk * D;
    const float* skb = sk_addrs[b] + hk;                      // (len_buf, H_kv)
    const float* svb = sv_addrs[b] + hk;

    const int8_t* mrow = nullptr;
    if (mask) {
        size_t len_off = 0;
        for (int j = 0; j < b; ++j) len_off += buf_lens[j];
        mrow = mask + (size_t)len_q * len_off + (size_t)qi * len_buf;
    }

    // ---- phase 1: S = K.Q^T on tensor cores (K bytes -> exact fp16 integers) ----
    uint4 qf[NI];
#pragma unroll
    for (int i = 0; i < NI; ++i)
        qf[i] = (g < mq) ? ld_cg_u4(q + ((size_t)bq * num_heads + head0 + g) * D + i * 32 + t * 8) : make_uint4(0, 0, 0, 0);
    const int ntiles = (n + 15) >> 4;
    for (int tile = warp; tile < ntiles; tile += kA8Warps) {
        const int ka_i = k0 + tile * 16 + g, kb_i = ka_i + 8;
        const int ra = min(ka_i, k1 - 1), rb = min(kb_i, k1 - 1);
        const uint8_t* pa = kbase + (size_t)ra * stride + t * 8;
        const uint8_t* pb = kbase + (size_t)rb * stride + t * 8;
        uint2 ka[NI], kb[NI];
#pragma unroll
        for (int i = 0; i < NI; ++i) {
            ka[i] = ld_cg_b8(pa + i * 32);
            kb[i] = ld_cg_b8(pb + i * 32);
        }
        const float sa = __ldcg(skb + (size_t)ra * num_kv_heads), sb = __ldcg(skb + (size_t)rb * num_kv_heads);
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int i = 0; i < NI; ++i) {
            uint32_t a01, a23, a45, a67, b01, b23, b45, b67;
            u8x4_to_h2x2(ka[i].x, a01, a23);
            u8x4_to_h2x2(ka[i].y, a45, a67);
            u8x4_to_h2x2(kb[i].x, b01, b23);
            u8x4_to_h2x2(kb[i].y, b45, b67);
            const uint32_t f0[4] = {a01, b01, a23, b23};
            const uint32_t f1[4] = {a45, b45, a67, b67};
            mma_16816_f16(acc, f0, qf[i].x, qf[i].y, acc);
            mma_16816_f16(acc, f1, qf[i].z, qf[i].w, acc);
        }
        const bool va = ka_i < k1 && (!mrow || mrow[ka_i] != 0);
        const bool vb = kb_i < k1 && (!mrow || mrow[kb_i] != 0);
        const int la = tile * 16 + g;
        const float ninf = -INFINITY;
        if (2 * t < mq) {
            s_logit[(2 * t) * kA8RowStride + la] = va ? acc[0] * sa * scale : ninf;
            s_logit[(2 * t) * kA8RowStride + la + 8] = vb ? acc[2] * sb * scale : ninf;
        }
        if (2 * t + 1 < mq) {
            s_logit[(2 * t + 1) * kA8RowStride + la] = va ? acc[1] * sa * scale : ninf;
            s_logit[(2 * t + 1) * kA8RowStride + la + 8] = vb ? acc[3] * sb * scale : ninf;
        }
    }
    __syncthreads();

    // ---- phase 2: masked softmax statistics per head; the V scale is folded into the stored weights ----
    for (int h = warp; h < mq; h += kA8Warps) {
        float* row = s_logit + h * kA8RowStride;
        float mx = -1e20f;
        for (int i = lane; i < n; i += 32) mx = fmaxf(mx, row[i]);
        mx = warp_max(mx);
        float sum = 0.f, svmax = 0.f;
        for (int i = lane; i < n; i += 32) {
            const float e = expf(row[i] - mx);
            const float sv = __ldcg(svb + (size_t)(k0 + i) * num_kv_heads);
            sum += e;
            svmax = fmaxf(svmax, fabsf(sv));
            row[i] = e * sv;
        }
        sum = warp_sum(sum) + 1e-20f;
        svmax = warp_max(svmax);
        if (lane == 0) {
            s_m[h] = mx;
            s_l[h] = sum;
            if (h == 0) {
                int ex;
                frexpf(svmax, &ex);                  // svmax = m 2^ex, m in [0.5, 1)  (svmax = 0: ex = 0)
                s_wexp = max(ex, -116);              // keeps 2^(10 - ex) and 2^(ex - 10) normal floats
            }
        }
    }
    __syncthreads();

    // ---- phase 3: O = (P * scale_v) . (V - 128) on the tensor cores (mma.sync m16n8k16, fp32 accumulate) ----
    // A = weights [head (8 of 16 rows) x 16 keys] as fp16, scaled by 2^(10 - ex) where 2^ex bounds the largest V scale of the
    // CTA's keys: every weight is p * scale_v <= scale_v, so the largest lands below 1024 (no fp16 overflow for any V
    // magnitude) and near it (small weights stay normal numbers); the power of two is undone exactly at write-out.
    // B = V [16 keys x 8 columns] as exact fp16 integers.  A B fragment register holds TWO KEYS of one column, V is stored
    // key-major: lane (g, t) loads D/8 contiguous bytes (columns NJ g .. NJ g + NJ - 1) of its four keys 2t, 2t+1, 2t+8,
    // 2t+9 and byte-interleaves row pairs with PRMT; n-tile j column c then stands for column d = NJ c + j of V (any
    // permutation of the columns is as good as another -- it is undone when the accumulators are written out).
    constexpr int NJ = D / 8;                        // n-tiles = V columns per lane and key row
    constexpr int NW = NJ / 4;                       // 32-bit words of a lane's column chunk
    float o[NJ][4];
#pragma unroll
    for (int j = 0; j < NJ; ++j) o[j][0] = o[j][1] = o[j][2] = o[j][3] = 0.f;
    const __half2 voff = __float2half2_rn(1152.f);   // 1024 (magic) + 128 (zero point of the cache)
    const float wscale = ldexpf(1.f, 10 - s_wexp);
    for (int tile = warp; tile < ntiles; tile += kA8Warps) {
        const int kb = tile * 16;                    // first key of the tile, relative to k0
        uint32_t vw[4][NW];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int kk = kb + 2 * t + (r & 1) + (r >> 1) * 8;
#pragma unroll
            for (int w = 0; w < NW; ++w) vw[r][w] = 0x80808080u;          // out of range: v - 128 = 0
            if (kk < n) {
                const uint8_t* src = vbase + (size_t)(k0 + kk) * stride + g * NJ;
                if constexpr (NW == 4) {
                    const uint4 v = ld_cg_u4(src);
                    vw[r][0] = v.x, vw[r][1] = v.y, vw[r][2] = v.z, vw[r][3] = v.w;
                } else {
                    const uint2 v = ld_cg_b8(src);
                    vw[r][0] = v.x, vw[r][1] = v.y;
                }
            }
        }
        uint32_t af[4] = {0u, 0u, 0u, 0u};
        if (g < mq) {
            const float* pr = s_logit + g * kA8RowStride + kb + 2 * t;
            const float2 p0 = *reinterpret_cast<const float2*>(pr), p1 = *reinterpret_cast<const float2*>(pr + 8);
            const bool in0 = kb + 2 * t < n, in1 = kb + 2 * t + 1 < n, in2 = kb + 2 * t + 8 < n, in3 = kb + 2 * t + 9 < n;
            const __half2 h0 = __floats2half2_rn(in0 ? p0.x * wscale : 0.f, in1 ? p0.y * wscale : 0.f);
            const __half2 h1 = __floats2half2_rn(in2 ? p1.x * wscale : 0.f, in3 ? p1.y * wscale : 0.f);
            af[0] = *reinterpret_cast<const uint32_t*>(&h0);   // (head g, keys 2t, 2t+1)
            af[2] = *reinterpret_cast<const uint32_t*>(&h1);   // (head g, keys 2t+8, 2t+9); rows g+8 (a1, a3) stay zero
        }
#pragma unroll
        for (int wq = 0; wq < NW; ++wq) {
            // bytes 4 wq .. 4 wq + 3 of the key pairs -> {k, k+1} interleaved
            const uint32_t lo01 = __byte_perm(vw[0][wq], vw[1][wq], 0x5140), hi01 = __byte_perm(vw[0][wq], vw[1][wq], 0x7362);
            const uint32_t lo23 = __byte_perm(vw[2][wq], vw[3][wq], 0x5140), hi23 = __byte_perm(vw[2][wq], vw[3][wq], 0x7362);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const uint32_t s01 = e < 2 ? lo01 : hi01, s23 = e < 2 ? lo23 : hi23;
                const uint32_t sel = (e & 1) ? 0x4342u : 0x4140u;
                uint32_t b0 = __byte_perm(s01, 0x64646464u, sel), b1 = __byte_perm(s23, 0x64646464u, sel);
                __half2 hb0 = __hsub2(*reinterpret_cast<__half2*>(&b0), voff), hb1 = __hsub2(*reinterpret_cast<__half2*>(&b1), voff);
                mma_16816_f16(o[wq * 4 + e], af, *reinterpret_cast<uint32_t*>(&hb0), *reinterpret_cast<uint32_t*>(&hb1), o[wq * 4 + e]);
            }
        }
    }
    __syncthreads();
    float* s_red = s_logit;   // [warp][h][D]
    if (g < mq) {
        // accumulator (n-tile j, column c = 2t + i) = head g, V column NJ c + j; rows g + 8 (o[j][2..3]) are padding
        const float wunscale = ldexpf(1.f, s_wexp - 10);
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            s_red[(warp * 8 + g) * D + NJ * (2 * t) + j] = o[j][0] * wunscale;
            s_red[(warp * 8 + g) * D + NJ * (2 * t + 1) + j] = o[j][1] * wunscale;
        }
    }
    __syncthreads();
    for (int e = tid; e < mq * D; e += kA8Threads) {
        const int h = e / D, d = e % D;
        float v = 0.f;
#pragma unroll
        for (int w = 0; w < kA8Warps; ++w) v += s_red[(w * 8 + h) * D + d];
        v = v / s_l[h];
        const size_t vh = (size_t)bq * num_heads + head0 + h;
        if (num_splits == 1) {
            out[vh * D + d] = from_f32<TO>(v);
        } else {
            part_o[(vh * num_splits + split) * D + d] = v;
            if (d == 0) {
                part_m[vh * num_splits + split] = s_m[h];
                part_l[vh * num_splits + split] = s_l[h];
            }
        }
    }
}

// grid (B*len_q*num_heads), block D: LSE combine of the splits (attention_kernel.cu:881-923)
template <typename TO>
__global__ void k_attn_combine_kv8(const float* __restrict__ part_o, const float* __restrict__ part_m,
                                   const float* __restrict__ part_l, TO* __restrict__ out, int num_splits) {
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
    for (int i = 0; i < num_splits; ++i) res += part_o[((size_t)vh * num_splits + i) * D + d] * (pl[i] / gs * expf(pm[i] - gm));
    out[(size_t)vh * D + d] = from_f32<TO>(res);
}

// quant_calc_scale(x, 127, 128) of one (token, kv head) row + scatter into the task's cache at placement (BSHD):
// grid (B * len_q, H_kv, 2 [k, v]), block d
template <typename T>
__global__ void k_kv8_quant_append(const T* __restrict__ k_src, const T* __restrict__ v_src, const int32_t* __restrict__ token_batch,
                                   const int32_t* __restrict__ placement, uint8_t* const* __restrict__ k_addrs,
                                   uint8_t* const* __restrict__ v_addrs, float* const* __restrict__ sk_addrs,
                                   float* const* __restrict__ sv_addrs, int num_kv_heads) {
    __shared__ float s_max[32];
    const int tok = blockIdx.x, hk = blockIdx.y, is_v = blockIdx.z, d = blockDim.x, c = threadIdx.x;
    pdl_trigger();
    pdl_wait();
    const T* src = (is_v ? v_src : k_src) + ((size_t)tok * num_kv_heads + hk) * d;
    const float x = to_f32<T>(src[c]);
    float amax = warp_max(fabsf(x));
    if ((c & 31) == 0) s_max[c >> 5] = amax;
    __syncthreads();
    amax = 0.f;
    for (int w = 0; w < (d + 31) / 32; ++w) amax = fmaxf(amax, s_max[w]);
    const int pl = placement[tok];
    if (pl < 0) return;
    const int b = token_batch[tok];
    const float block_scale = 127.0f / amax;                      // quant_kernel.cu:31
    const float r = nearbyintf(x * block_scale);
    uint8_t* dst = (is_v ? v_addrs : k_addrs)[b] + ((size_t)pl * num_kv_heads + hk) * d;
    dst[c] = (uint8_t)(128.f + r);
    if (c == 0) (is_v ? sv_addrs : sk_addrs)[b][(size_t)pl * num_kv_heads + hk] = amax / 127.0f;
}

// dense form of the same quantisation: int8_op::quant_calc_scale(x, 127, 128) on (M, K) rows -> uint8 codes + fp32 scales
template <typename T>
__global__ void k_int8_quant_rows_u8(const T* __restrict__ x, uint8_t* __restrict__ q, float* __restrict__ scale, int K) {
    __shared__ float s_max[32];
    const size_t off = (size_t)blockIdx.x * K;
    float amax = 0.f;
    for (int i = threadIdx.x; i < K; i += blockDim.x) amax = fmaxf(amax, fabsf(to_f32<T>(x[off + i])));
    amax = warp_max(amax);
    if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = amax;
    __syncthreads();
    amax = 0.f;
    for (int w = 0; w < (int)(blockDim.x + 31) / 32; ++w) amax = fmaxf(amax, s_max[w]);
    const float block_scale = 127.0f / amax;
    for (int i = threadIdx.x; i < K; i += blockDim.x)
        q[off + i] = (uint8_t)(128.f + nearbyintf(to_f32<T>(x[off + i]) * block_scale));
    if (threadIdx.x == 0) scale[blockIdx.x] = amax / 127.0f;
}

}  // namespace zl

using namespace zl;

extern "C" int zl_int8_quant_rows_u8(const void* x, void* q, float* scale, int M, int K, int dtype, zl_stream_t stream) {
    ZL_CHECK_ARG(x && q && scale && M > 0 && K > 0);
    ZL_CHECK_SUPPORTED(dtype == ZL_F16 || dtype == ZL_BF16);
    const int threads = K >= 1024 ? 1024 : ((K + 31) / 32) * 32;
    if (dtype == ZL_F16)
        k_int8_quant_rows_u8<__half><<<M, threads, 0, stream>>>((const __half*)x, (uint8_t*)q, scale, K);
    else
        k_int8_quant_rows_u8<__nv_bfloat16><<<M, threads, 0, stream>>>((const __nv_bfloat16*)x, (uint8_t*)q, scale, K);
    ZL_CHECK_LAUNCH();
    return ZL_OK;
}

extern "C" int zl_kv_int8_quant_append(const void* k_src, const void* v_src, const int32_t* token_batch,
                                       const int32_t* placement, void* const* k_addrs, void* const* v_addrs,
                                       void* const* scale_k_addrs, void* const* scale_v_addrs, int T, int num_kv_heads,
                                       int dim_head, int dtype, int pdl, zl_stream_t stream) {
    ZL_CHECK_ARG(k_src && v_src && token_batch && placement && k_addrs && v_addrs && scale_k_addrs && scale_v_addrs);
    ZL_CHECK_ARG(T > 0 && num_kv_heads > 0 && dim_head > 0 && dim_head <= 1024 && dim_head % 32 == 0);
    ZL_CHECK_SUPPORTED(dtype == ZL_F16 || dtype == ZL_BF16);
    dim3 grid(T, num_kv_heads, 2), block(dim_head);
    if (dtype == ZL_F16)
        ZL_CHECK_CUDA(launch(k_kv8_quant_append<__half>, grid, block, 0, stream, pdl != 0, (const __half*)k_src,
                             (const __half*)v_src, token_batch, placement, (uint8_t* const*)k_addrs, (uint8_t* const*)v_addrs,
                             (float* const*)scale_k_addrs, (float* const*)scale_v_addrs, num_kv_heads));
    else
        ZL_CHECK_CUDA(launch(k_kv8_quant_append<__nv_bfloat16>, grid, block, 0, stream, pdl != 0, (const __nv_bfloat16*)k_src,
                             (const __nv_bfloat16*)v_src, token_batch, placement, (uint8_t* const*)k_addrs,
                             (uint8_t* const*)v_addrs, (float* const*)scale_k_addrs, (float* const*)scale_v_addrs,
                             num_kv_heads));
    return ZL_OK;
}

extern "C" int zl_decode_attention_kv8(const void* q, const int32_t* buf_lens, void* const* k_addrs, void* const* v_addrs,
                                       void* const* scale_k_addrs, void* const* scale_v_addrs, const int8_t* mask,
                                       float scale, int max_len_buf, void* out, int B, int len_q, int num_heads,
                                       int num_kv_heads, int dim_head, void* workspace, size_t workspace_bytes,
                                       int out_dtype, int pdl, zl_stream_t stream) {
    ZL_CHECK_ARG(q && buf_lens && k_addrs && v_addrs && scale_k_addrs && scale_v_addrs && out);
    ZL_CHECK_ARG(B > 0 && len_q > 0 && max_len_buf > 0 && num_heads > 0 && num_kv_heads > 0 && num_heads % num_kv_heads == 0);
    ZL_CHECK_SUPPORTED(dim_head == 128 || dim_head == 64);     // the reference: 128 only (attention_kernel.cu:1314)
    ZL_CHECK_SUPPORTED(out_dtype == ZL_F16 || out_dtype == ZL_BF16);
    const int m_query = num_heads / num_kv_heads;
    const int hgroups = (m_query + 7) / 8;
    const int base = B * len_q * num_kv_heads * hgroups;
    int splits = cdiv(2 * device_sm_count(), base);
    const int max_useful = cdiv(max_len_buf, 256);
    if (splits > max_useful) splits = max_useful;
    if (splits > kA8MaxSplits) splits = kA8MaxSplits;
    const int min_splits = cdiv(max_len_buf, kA8MaxRange);   // a CTA holds at most 1024 logits: may exceed kA8MaxSplits
    if (splits < min_splits) splits = min_splits;
    if (splits < 1) splits = 1;
    const size_t vheads = (size_t)B * len_q * num_heads;
    float *part_o = nullptr, *part_m = nullptr, *part_l = nullptr;
    if (splits > 1) {
        const size_t need = vheads * splits * (dim_head + 2) * sizeof(float);
        ZL_CHECK_ARG(workspace != nullptr && workspace_bytes >= need);
        part_o = static_cast<float*>(workspace);
        part_m = part_o + vheads * splits * dim_head;
        part_l = part_m + vheads * splits;
    }
    dim3 grid(splits, num_kv_heads * hgroups, B * len_q), block(kA8Threads);
#define ZL_A8_LAUNCH(TO, DD)                                                                                         \
    ZL_CHECK_CUDA(launch(k_decode_attn_kv8<TO, DD>, grid, block, 0, stream, pdl != 0, (const __half*)q, buf_lens,    \
                         (uint8_t* const*)k_addrs, (uint8_t* const*)v_addrs, (float* const*)scale_k_addrs,           \
                         (float* const*)scale_v_addrs, mask, scale, (TO*)out, part_o, part_m, part_l, len_q,         \
                         num_heads, num_kv_heads, m_query, splits));                                                 \
    if (splits > 1)                                                                                                  \
        ZL_CHECK_CUDA(launch(k_attn_combine_kv8<TO>, dim3((unsigned)vheads), dim3(DD), 0, stream, pdl != 0,          \
                             (const float*)part_o, (const float*)part_m, (const float*)part_l, (TO*)out, splits));
    if (out_dtype == ZL_F16) {
        if (dim_head == 128) { ZL_A8_LAUNCH(__half, 128) } else { ZL_A8_LAUNCH(__half, 64) }
    } else {
        if (dim_head == 128) { ZL_A8_LAUNCH(__nv_bfloat16, 128) } else { ZL_A8_LAUNCH(__nv_bfloat16, 64) }
    }
#undef ZL_A8_LAUNCH
    return ZL_OK;
}
