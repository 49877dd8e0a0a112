// Kernel parameter block of the W4A16 GEMM variants (host + device).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace zl {

struct W4Params {
    const __half* x;
    int ldx;
    const uint8_t* packed;
    const __half* bias;       // indexed by PACKED row
    const __half* residual;
    __half* y;
    int mc, N, K, epi;
    // fused RMSNorm prologue (ln_w == nullptr: off)
    const __half* ln_w;
    float eps;
    // ZL_EPI_QKV_ROPE
    const float* cos;
    const float* sin;
    __half* q_out;
    const int32_t* token_batch;
    const int32_t* placement;
    __half* const* k_addrs;
    __half* const* v_addrs;
    int num_heads, num_kv_heads, dim_head;
    // weights of the NEXT kernel in the chain: prefetched into L2 when this CTA runs out of work (may be null)
    const uint8_t* pf_ptr;
    unsigned long long pf_bytes;
    unsigned long long* trace;   // debug: per-CTA globaltimer samples [grid][16] (zl_w4_set_trace)
    int dbg;   // ZL_W4_DEBUG: 1 = skip dequant/MMA (pure weight-stream probe; results are garbage)
    // tensor-parallel exchange inside the GEMM (integer kernel only; comm_dev.cuh).  tp_mode 1 (reduce-in): the
    // activation row is  T(T(sum over ranks of the partial sums pushed by the previous row-parallel GEMM) + x)  -- x is the
    // residual stream -- and CTA 0 stores it to tp_h_out (must not alias x).  tp_mode 2 (push): the epilogue stores the
    // fp16 partial tile into every rank's inbox and the last CTA publishes the epoch flags.
    const void* tp_cd = nullptr;   // const CommDev*
    int tp_mode = 0;
    int tp_index = 0;              // exchange index within the step (< 512): parity of the slot + part of the word tag
    __half* tp_h_out = nullptr;
};

cudaError_t launch_w4_v2(const W4Params& p, bool pdl, cudaStream_t stream);
cudaError_t prepare_w4_v2();
// exact-integer kernel on the ZLW4I layout; false = staged activations do not fit shared memory
bool launch_w4_v3(const W4Params& p, bool pdl, cudaStream_t stream, cudaError_t* err);
bool w4_v3_fits(int mc, int N, int K);
cudaError_t prepare_w4_v3();
// tcgen05 / TMEM / TMA kernel on the ZLW4I layout (w4a16_tc.cu): up to 256 tokens per launch, N % 128 == 0, no fused
// RMSNorm prologue (ln_w is ignored)
cudaError_t launch_w4_tc(const W4Params& p, bool pdl, cudaStream_t stream);
bool w4_tc_supports(int mc, int N, int K);
cudaError_t prepare_w4_tc();
cudaError_t prepare_w8_tc();   // w8_tc.cu
cudaError_t prepare_sample();  // sample.cu

}  // namespace zl
