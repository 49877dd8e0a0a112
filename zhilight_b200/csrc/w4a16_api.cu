// Front end of the W4A16 Linear (C-ABI): kernel selection by M, packing row maps, one-time preparation.
//
// Stands in for nn::gptq::gptq_gemm_k_major's router (reference src/nn/quant/gptq/q_gemm_k_major.cu:957-1116:
// M <= 40 GEMV, else dequant + cuBLASLt) and for GPTQMarlin::forward (src/nn/linear/linear.cpp:1247-1451):
//   M <= 16 and the staged activations fit shared memory -> k_w4a16_v3  (exact-integer mma.sync kernel, ZLW4I layout)
//   otherwise, N % 128 == 0                              -> k_w4a16_ts  (tcgen05 kernel, A operand in TMEM, ZLW4I layout)
//   otherwise                                            -> k_w4a16_v2  (fp16 mma.sync kernel, ZLW4 layout, 32-row passes)
#include "common.cuh"
#include "w4_layout.cuh"
#include "w4_params.h"
#include "comm_dev.cuh"

#include <cstdlib>

using namespace zl;

extern "C" int zl_prepare(void) {
    // opt-in shared memory sizes and the per-device split-k workspace of the tcgen05 kernel must be set up outside of
    // stream capture; idempotent per device
    ZL_CHECK_CUDA(prepare_w4_v2());
    ZL_CHECK_CUDA(prepare_w4_v3());
    ZL_CHECK_CUDA(prepare_w4_tc());
    ZL_CHECK_CUDA(prepare_w8_tc());
    ZL_CHECK_CUDA(prepare_sample());
    return ZL_OK;
}

// ZL_W4_NO_TC=1 (experiments): never route to the tcgen05 kernel
static bool tc_disabled() {
    static int v = -1;
    if (v < 0) v = getenv("ZL_W4_NO_TC") ? 1 : 0;
    return v != 0;
}

// which kernel serves (M, N, K) on the ZLW4I layout: 3 = exact-integer mma.sync, 4 = tcgen05, 0 = neither
static int int_layout_route(int M, int N, int K) {
    if (M <= 16 && w4_v3_fits(M, N, K)) return 3;
    if (!tc_disabled() && w4_tc_supports(M < 256 ? M : 256, N, K)) return 4;
    return 0;
}

namespace zl {
__global__ void k_qkv_rope_row_map(int32_t* map, int n_rows, int d) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_rows) return;
    const int tiles_per_head = d / 32;
    const int st = p >> 5, head = st / tiles_per_head, jt = st % tiles_per_head;
    const int r32 = p & 31, tt = r32 >> 4, r16 = r32 & 15;
    const int c = jt * 16 + tt * 8 + (r16 & 7);
    map[p] = head * d + c + ((r16 >= 8) ? d / 2 : 0);
}
__global__ void k_gather_16(const uint16_t* __restrict__ src, const int32_t* __restrict__ map, uint16_t* __restrict__ dst,
                            int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = src[map[i]];
}
}  // namespace zl

unsigned long long* g_w4_trace = nullptr;   // shared with dense_gemm.cu (per-launch timeline records)
extern "C" int zl_w4_set_trace(void* buf) {
    g_w4_trace = static_cast<unsigned long long*>(buf);
    return ZL_OK;
}

extern "C" int zl_w4_int_kernel_fits(int M, int N, int K) {
    if (M <= 0 || N <= 0 || K <= 0 || N % 32 || K % kW4GroupK) return 0;
    return (M <= 16 && w4_v3_fits(M, N, K)) ? 1 : 0;
}

extern "C" int zl_w4_int_layout_route(int M, int N, int K) {
    if (M <= 0 || N <= 0 || K <= 0 || N % 32 || K % kW4GroupK) return 0;
    return int_layout_route(M, N, K);
}

extern "C" int zl_qkv_rope_row_map(int32_t* row_map, int n_heads_total, int dim_head, zl_stream_t stream) {
    ZL_CHECK_ARG(row_map && n_heads_total > 0 && dim_head > 0);
    ZL_CHECK_SUPPORTED(dim_head % 32 == 0);
    const int n = n_heads_total * dim_head;
    k_qkv_rope_row_map<<<cdiv(n, 256), 256, 0, stream>>>(row_map, n, dim_head);
    ZL_CHECK_LAUNCH();
    return ZL_OK;
}

extern "C" int zl_gather_rows_16(const void* src, const int32_t* map, void* dst, int n, zl_stream_t stream) {
    ZL_CHECK_ARG(src && map && dst && n > 0);
    k_gather_16<<<cdiv(n, 256), 256, 0, stream>>>((const uint16_t*)src, map, (uint16_t*)dst, n);
    ZL_CHECK_LAUNCH();
    return ZL_OK;
}

extern "C" int zl_w4a16_gemm_fused(const zl_w4_fused_args_t* a, zl_stream_t stream) {
    {
        static bool prepared[64] = {};
        int dev = 0;
        cudaGetDevice(&dev);
        if (dev < 0 || dev >= 64 || !prepared[dev]) {
            int rc = zl_prepare();
            if (rc != ZL_OK) return rc;
            if (dev >= 0 && dev < 64) prepared[dev] = true;
        }
    }
    ZL_CHECK_ARG(a && a->x && a->packed && a->M > 0 && a->N > 0 && a->K > 0);
    ZL_CHECK_SUPPORTED(a->group_size == kW4GroupK);
    ZL_CHECK_SUPPORTED(a->N % 32 == 0 && a->K % kW4GroupK == 0);
    ZL_CHECK_ARG(a->ldx >= a->K && a->ldx % 8 == 0);
    ZL_CHECK_ARG((reinterpret_cast<uintptr_t>(a->x) & 15) == 0 && (reinterpret_cast<uintptr_t>(a->packed) & 15) == 0);
    ZL_CHECK_ARG(a->epilogue >= ZL_EPI_NONE && a->epilogue <= ZL_EPI_QKV_ROPE);
    ZL_CHECK_ARG(a->variant == kW4VariantHalf || a->variant == kW4VariantInt);
    ZL_CHECK_ARG(a->epilogue != ZL_EPI_RESIDUAL || a->residual != nullptr);
    ZL_CHECK_ARG(a->epilogue == ZL_EPI_QKV_ROPE || a->y != nullptr || a->tp_mode == 2);
    ZL_CHECK_ARG(a->ln_weight == nullptr || (reinterpret_cast<uintptr_t>(a->ln_weight) & 15) == 0);
    if (a->epilogue == ZL_EPI_QKV_ROPE) {
        ZL_CHECK_ARG(a->cos && a->sin && a->q_out && a->token_batch && a->placement && a->k_addrs && a->v_addrs);
        ZL_CHECK_ARG(a->num_heads > 0 && a->num_kv_heads > 0 && a->dim_head > 0);
        ZL_CHECK_SUPPORTED(a->dim_head % 32 == 0);
        ZL_CHECK_ARG(a->N == (a->num_heads + 2 * a->num_kv_heads) * a->dim_head);
    }
    const void* tp_cd = nullptr;
    if (a->tp_mode != 0) {
        ZL_CHECK_ARG(a->tp_mode == 1 || a->tp_mode == 2);
        ZL_CHECK_ARG(a->tp_index >= 0 && a->tp_index < 1024);
        ZL_CHECK_ARG(a->tp_comm != nullptr && a->variant == kW4VariantInt);
        tp_cd = zl_comm_device_state(a->tp_comm);
        if (!tp_cd) {
            zl_set_last_error(__FILE__, __LINE__, "tp_comm: peers not opened");
            return ZL_ERR_STATE;
        }
        ZL_CHECK_SUPPORTED(a->M <= 16 && w4_v3_fits(a->M, a->N, a->K) && "tp_mode needs the integer kernel (M <= 16)");
        if (a->tp_mode == 1) {
            ZL_CHECK_ARG(a->tp_h_out != nullptr && a->tp_h_out != a->x && a->ldx == a->K);
            ZL_CHECK_ARG((size_t)a->M * a->K * 2 <= zl_comm_slot_bytes(a->tp_comm));
        } else {
            ZL_CHECK_ARG(a->epilogue == ZL_EPI_NONE && a->bias == nullptr);
            ZL_CHECK_ARG((size_t)a->M * a->N * 2 <= zl_comm_slot_bytes(a->tp_comm));
        }
    }
    const int n_out = a->epilogue == ZL_EPI_SWIGLU ? a->N / 2 : a->N;
    // rows per pass: the tcgen05 kernel takes up to 256 tokens at once, the mma.sync kernels 32 (v2) / 16 (v3)
    const int route = a->variant == kW4VariantInt ? int_layout_route(a->M, a->N, a->K) : 2;
    ZL_CHECK_SUPPORTED(route != 0 && "ZLW4I layout: M > 16 (or staged activations too large) and N % 128 != 0: use variant 0");
    ZL_CHECK_SUPPORTED(!(route == 4 && a->ln_weight) && "the tcgen05 kernel has no fused RMSNorm prologue: run zl_rmsnorm first");
    const int step = route == 4 ? 256 : 32;
    for (int m0 = 0; m0 < a->M; m0 += step) {
        W4Params p;
        p.mc = (a->M - m0) < step ? (a->M - m0) : step;
        p.x = static_cast<const __half*>(a->x) + (size_t)m0 * a->ldx;
        p.ldx = a->ldx;
        p.packed = static_cast<const uint8_t*>(a->packed);
        p.bias = static_cast<const __half*>(a->bias);
        p.residual = a->residual ? static_cast<const __half*>(a->residual) + (size_t)m0 * a->N : nullptr;
        p.y = a->y ? static_cast<__half*>(a->y) + (size_t)m0 * n_out : nullptr;
        p.N = a->N;
        p.K = a->K;
        p.epi = a->epilogue;
        p.ln_w = static_cast<const __half*>(a->ln_weight);
        p.eps = a->eps;
        p.cos = a->cos ? a->cos + (size_t)m0 * a->dim_head : nullptr;
        p.sin = a->sin ? a->sin + (size_t)m0 * a->dim_head : nullptr;
        p.q_out = a->q_out ? static_cast<__half*>(a->q_out) + (size_t)m0 * a->num_heads * a->dim_head : nullptr;
        p.token_batch = a->token_batch ? a->token_batch + m0 : nullptr;
        p.placement = a->placement ? a->placement + m0 : nullptr;
        p.k_addrs = reinterpret_cast<__half* const*>(a->k_addrs);
        p.v_addrs = reinterpret_cast<__half* const*>(a->v_addrs);
        p.num_heads = a->num_heads;
        p.num_kv_heads = a->num_kv_heads;
        p.dim_head = a->dim_head;
        {
            static int dbg = -1;
            if (dbg < 0) {
                const char* e = getenv("ZL_W4_DEBUG");
                dbg = e ? atoi(e) : 0;
            }
            p.dbg = dbg;
        }
        p.trace = g_w4_trace;
        if (p.dbg & 32) p.ln_w = nullptr;   // timing probe: drop the fused RMSNorm (results are wrong)
        p.tp_cd = tp_cd;
        p.tp_mode = a->tp_mode;
        p.tp_index = a->tp_index;
        p.tp_h_out = static_cast<__half*>(a->tp_h_out);
        p.pf_ptr = static_cast<const uint8_t*>(a->prefetch_ptr);
        p.pf_bytes = a->prefetch_bytes;
        if (route == 4) {
            ZL_CHECK_CUDA(launch_w4_tc(p, a->pdl != 0 && m0 == 0, stream));
        } else if (route == 3) {
            cudaError_t ce = cudaSuccess;
            const bool ok = launch_w4_v3(p, a->pdl != 0 && m0 == 0, stream, &ce);
            ZL_CHECK_SUPPORTED(ok && "ZLW4I kernel: staged activations do not fit shared memory (use variant 0)");
            ZL_CHECK_CUDA(ce);
        } else {
            ZL_CHECK_CUDA(launch_w4_v2(p, a->pdl != 0 && m0 == 0, stream));
        }
    }
    return ZL_OK;
}

extern "C" int zl_w4a16_gemm(const void* x, int ldx, const void* packed, const void* bias, const void* residual,
                             void* y, int M, int N, int K, int group_size, int epilogue, int pdl,
                             zl_stream_t stream) {
    ZL_CHECK_ARG(x && packed && y && M > 0 && N > 0 && K > 0);
    ZL_CHECK_SUPPORTED(group_size == kW4GroupK);
    ZL_CHECK_SUPPORTED(N % 32 == 0 && K % kW4GroupK == 0);
    ZL_CHECK_ARG(ldx >= K && ldx % 8 == 0);
    ZL_CHECK_ARG((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(packed) & 15) == 0);
    ZL_CHECK_ARG(epilogue == ZL_EPI_NONE || epilogue == ZL_EPI_SWIGLU || epilogue == ZL_EPI_RESIDUAL);
    ZL_CHECK_ARG(epilogue != ZL_EPI_RESIDUAL || residual != nullptr);
    zl_w4_fused_args_t a = {};
    a.x = x; a.ldx = ldx; a.packed = packed; a.bias = bias; a.residual = residual; a.y = y;
    a.M = M; a.N = N; a.K = K; a.group_size = group_size; a.epilogue = epilogue; a.pdl = pdl;
    return zl_w4a16_gemm_fused(&a, stream);
}
