/*
 * zhilight_b200 -- C-ABI of the B200-native (sm_100a) quantized-decode hot path of ZhiLight.
 *
 * Every entry point replaces one reference operator (cited as file:line under /root/reference).
 * Conventions (SURVEY.md section 8b):
 *   - plain pointers + sizes, no C++/torch types; all data pointers are DEVICE pointers unless
 *     the name ends in _host;
 *   - stream-ordered on `stream`, no allocation, no host sync inside (except zl_llama_* which
 *     owns its buffers);
 *   - returns ZL_OK (0) or a negative error code; zl_last_error() gives the message of the last
 *     failure on the calling thread.  The C++ mirror (zhilight_b200/host) turns codes into the
 *     reference's BMEngineException behaviour;
 *   - re-entrant per device; no global mutable state besides per-device symmetric buffers
 *     created by zl_comm_*.
 *
 * dtype codes follow bmengine core::DataType ordering where they overlap
 * (3rd/bmengine/bmengine/include/bmengine/core/dtype.h).
 */
#ifndef ZHILIGHT_B200_H_
#define ZHILIGHT_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* zl_stream_t; /* == cudaStream_t */

enum {
    ZL_OK = 0,
    ZL_ERR_INVALID_ARG = -1,
    ZL_ERR_UNSUPPORTED = -2,
    ZL_ERR_CUDA = -3,
    ZL_ERR_STATE = -4
};

enum { ZL_F16 = 0, ZL_BF16 = 1, ZL_F32 = 2 };

/* epilogues of zl_w4a16_gemm */
enum {
    ZL_EPI_NONE = 0,     /* y = acc (+bias)                                                     */
    ZL_EPI_SWIGLU = 1,   /* packed rows interleave gate/up; y[:, n] = silu(T(gate)) * T(up)      */
    ZL_EPI_RESIDUAL = 2, /* y = T(T(acc (+bias)) + residual)   (block_kernel.cu:7-17)           */
    ZL_EPI_QKV_ROPE = 3  /* fused qkv: split + RoPE(q,k) + KV append (zl_w4a16_gemm_fused only)    */
};

const char* zl_last_error(void);
int zl_version(void);
/* number of kernel launches issued by this library on the calling thread since the last reset */
long long zl_launch_count(int reset);
/* one-time per-device kernel attribute setup (opt-in shared memory); called by zl_llama_create and lazily
 * by the ops; must not first happen inside a stream capture. */
int zl_prepare(void);

/* ------------------------------------------------------------------------------------------ *
 * Load-time integer layout transforms (bit-exact with the reference)
 * ------------------------------------------------------------------------------------------ */
/* nn::gptq::gptq_shuffle  (src/nn/quant/gptq/q_gemm.cu:778-872, qdq_4.cuh:16-35).
 * qweight (K/8, N) int32 in place.  q_perm (K) int32 or NULL; scratch (K/8*N words) required iff q_perm. */
int zl_gptq_shuffle(uint32_t* qweight, const int32_t* q_perm, uint32_t* scratch, int K, int N,
                    zl_stream_t stream);
/* nn::gptq::increase_zero (src/nn/quant/gptq/utils.cu:61-88): each nibble (z+1)&15, in place. */
int zl_gptq_increase_zero(uint32_t* qzeros, size_t n_words, zl_stream_t stream);
/* nn::gptq::subtract8 (utils.cu:91-118). */
int zl_gptq_subtract8(uint32_t* words, size_t n_words, zl_stream_t stream);
/* nn::gptq::q4_to_q8 (utils.cu:177-214): (R, C/8) int32 -> (R, C) uint8. */
int zl_q4_to_q8(const uint32_t* in, uint8_t* out, size_t n_words, zl_stream_t stream);
/* nn::gptq::un_shuffle (utils.cu:25-58): AWQ zero de-interleave in place, (rows, cols) words. */
int zl_awq_un_shuffle(uint32_t* qzeros, int rows, int cols, zl_stream_t stream);
/* nn::gptq::shuffle_awq (utils.cu:121-174): (K, N/8) -> (K/8, N). */
int zl_awq_shuffle(const uint32_t* in, uint32_t* out, int K, int N, int use_exllama, zl_stream_t stream);
/* functions::Transpose for 2-D tensors of 1/2/4-byte elements: (rows, cols) -> (cols, rows). */
int zl_transpose_2d(const void* in, void* out, int rows, int cols, int elem_bytes, zl_stream_t stream);
/* nn::gptq::dequant_k_major out_type 0 (q_gemm_k_major.cu:843-905): W16[n,k] = half(q-z)*half(s). */
int zl_gptq_dequant_k_major(const uint32_t* qweight_km, const uint8_t* qzeros_km, const void* scales_km,
                            void* out_f16, int N, int K, int group_size, zl_stream_t stream);

/* ------------------------------------------------------------------------------------------ *
 * ZLW4: the B200 tile-packed W4 layout consumed by zl_w4a16_gemm (DESIGN.md section 3).
 * Built once at load from the reference k-major tensors
 * (Int4GPTQ::preprocess_weight, src/nn/linear/linear.cpp:1139-1160).
 * ------------------------------------------------------------------------------------------ */
size_t zl_w4_packed_bytes(int N, int K, int group_size);
/* qweight_km (N_src, K/8) u32 shuffled, qzeros_km (N_src, K/g) u8 (NULL or sym!=0 -> zero 8),
 * scales_km (N_src, K/g) f16.  row_map (N) int32 or NULL: packed row p takes source row row_map[p]. */
int zl_w4_pack(const uint32_t* qweight_km, const uint8_t* qzeros_km, const void* scales_km,
               const int32_t* row_map, void* packed, int N, int K, int group_size, int sym,
               zl_stream_t stream);
/* variant 0: ZLW4 (fp16 HMMA kernels); variant 1: ZLW4I (exact-integer IMMA kernel, zl_w4a16_gemm_fused with
 * args.variant = 1).  zl_w4_pack == variant 0. */
int zl_w4_pack_v(const uint32_t* qweight_km, const uint8_t* qzeros_km, const void* scales_km,
                 const int32_t* row_map, void* packed, int N, int K, int group_size, int sym, int variant,
                 zl_stream_t stream);
int zl_w4_unpack_v(const void* packed, uint32_t* qweight_km, uint8_t* qzeros_km, void* scales_km, int N, int K,
                   int group_size, int variant, zl_stream_t stream);
/* inverse (tests): recover k-major nibbles/zeros/scales from the packed form. */
int zl_w4_unpack(const void* packed, uint32_t* qweight_km, uint8_t* qzeros_km, void* scales_km, int N, int K,
                 int group_size, zl_stream_t stream);

/* nn::gptq::gptq_gemm_k_major / KERNEL_gemm_warp_reduce / gemm_fuse_gate_in
 * (src/nn/quant/gptq/q_gemm_k_major.cu:957-1116, 176-237, 529-578):
 * y[m,n] = sum_k x[m,k] * (q[n,k]-z[n,k/g]) * s[n,k/g] (+bias[n]), fp16 in/out, fp32 accumulate.
 * x (M, K) f16 row stride ldx; y (M, N_out) f16 where N_out = N (NONE/RESIDUAL) or N/2 (SWIGLU).
 * Any M >= 1 (weights are re-streamed per 32-token chunk).  pdl != 0 -> programmatic dependent launch. */
int zl_w4a16_gemm(const void* x, int ldx, const void* packed, const void* bias, const void* residual,
                  void* y, int M, int N, int K, int group_size, int epilogue, int pdl, zl_stream_t stream);

/* The same GEMM with the neighbouring operators of the decode layer folded in (DESIGN.md section 4.1):
 *   ln_weight != NULL : nn::LayerNorm (rms, layernorm.cu:9-42) of x is fused into the prologue:
 *                       y = rsqrt(mean(x^2)+eps) * (W . (x*ln_weight)) (+bias);
 *   epilogue ZL_EPI_QKV_ROPE: W is the fused qkv weight packed with zl_qkv_rope_row_map; the epilogue applies
 *                       rope_qk_cache (rotary_embedding_fuse_cache.cu:23-63) and copy_to_rag_buffer2
 *                       (ragged_buffer_kernel.cu:194-222, BSHD) and writes q (M, num_heads*dim_head).
 *   tp_mode (tensor parallel, integer kernel only; replaces ModelContext::reduce_sum + element_add_scale between a
 *                       row-parallel Linear and the next column-parallel one, model_context.cpp:203-243, block.cpp:123-141):
 *                       2 on the row-parallel GEMM (o_proj / w_out, epilogue NONE, y unused): the fp16 partial tile is
 *                       stored straight into every rank's NVLink-mapped inbox of tp_comm as 8-byte words {2 x fp16, tag}
 *                       (valid on arrival: no flags, no fences);
 *                       1 on the next GEMM: its activation row becomes T(T(sum_r partial_r) + x), x = residual stream,
 *                       reduced in rank order while the activations are staged (the staging loop polls the words' tags);
 *                       the sum is also stored to tp_h_out (M, K; must not alias x).  0: off.
 *                       tp_index: index of the exchange within the step (0 .. 511, consecutive, the same on producer and
 *                       consumer), | 512 when the step has an ODD number of exchanges (the two slots must alternate across
 *                       step boundaries too); zl_comm_ll_begin_step(tp_comm) must be enqueued once per step before the
 *                       first such GEMM, on every rank.
 * bias is indexed by PACKED row. */
typedef struct zl_comm zl_comm_t;
typedef struct zl_w4_fused_args {
    const void* x; int ldx; const void* packed; const void* bias; const void* residual; void* y;
    int M, N, K, group_size, epilogue, pdl;
    const void* ln_weight; float eps;
    const float* cos; const float* sin; void* q_out;
    const int32_t* token_batch; const int32_t* placement; void* const* k_addrs; void* const* v_addrs;
    int num_heads, num_kv_heads, dim_head;
    const void* prefetch_ptr; size_t prefetch_bytes; /* next kernel's weights: pulled into L2 as this one drains (may be NULL) */
    int variant; /* layout of `packed`: 0 ZLW4, 1 ZLW4I (integer kernel; needs the staged activations to fit smem) */
    zl_comm_t* tp_comm; int tp_mode; void* tp_h_out; int tp_index;
} zl_w4_fused_args_t;
int zl_w4a16_gemm_fused(const zl_w4_fused_args_t* args, zl_stream_t stream);
/* 1 if the exact-integer kernel (variant 1, M <= 16) can run this shape: its staged activations must fit shared memory. */
int zl_w4_int_kernel_fits(int M, int N, int K);
/* which kernel serves (M, N, K) on the ZLW4I layout (variant 1): 3 = exact-integer mma.sync kernel, 4 = tcgen05 / TMEM /
 * TMA kernel (any M, N % 128 == 0, no fused RMSNorm prologue), 0 = neither (pack variant 0 and use the fp16 mma.sync kernel). */
int zl_w4_int_layout_route(int M, int N, int K);
/* last watchdog code published by a tcgen05 kernel on the current device (0 = none); a bounded mbarrier wait that expires
 * records which pipeline barrier starved and traps instead of hanging the GPU. */
unsigned zl_w4_tc_watchdog(void);
/* debug / tests: at least `splits` pieces per weight-row tile in the tcgen05 kernel's stream-k schedule (0 = automatic; also
 * ZL_TC_SPLITS). */
int zl_w4_tc_set_splits(int splits);
/* tests: host view of the tcgen05 kernel's stream-k schedule (the kernel's own scheduling code): pieces of CTA `cta` of `ctas`
 * for n_tiles x G (tile, group) units; out[5 i ..] = tile, g0, g1, pieces of that tile, workspace slot (-1: whole tile);
 * returns the number of pieces. */
int zl_w4_tc_schedule(int n_tiles, int G, int ctas, int cta, int* out, int max_pieces);
/* debug: with ZL_TC_DBG & 16, CTA 0 of the tcgen05 kernel stamps its pipeline hand-overs with clock64; copies
 * [11 roles][64 stages][4 events] of the last launch to `out` (n <= 2816 values). */
int zl_w4_tc_read_trace(long long* out, int n);
/* debug: device buffer of grid*16 uint64 globaltimer samples written by the integer kernel (NULL = off). */
int zl_w4_set_trace(void* buf);
/* row_map (n_heads_total*dim_head) for zl_w4_pack so that RoPE partners (c, c+d/2) share an MMA tile. */
int zl_qkv_rope_row_map(int32_t* row_map, int n_heads_total, int dim_head, zl_stream_t stream);
/* dst[i] = src[map[i]] for 16-bit elements (bias permutation to packed-row order). */
int zl_gather_rows_16(const void* src, const int32_t* map, void* dst, int n, zl_stream_t stream);

/* ---- W8A8 Linear: SmoothQuant INT8 (Int8Linear, src/nn/linear/linear.cpp:432-636) and per-tensor FP8 e4m3
 * (Fp8Linear, linear.cpp:1612-1695) ---------------------------------------------------------------------- */
enum { ZL_W8_INT8 = 0, ZL_W8_FP8 = 1, ZL_W8_FP8_ROWS = 2 /* fp8 with one f32 weight scale per output row */ };
/* int8_op::quant_calc_scale (src/nn/quant/int8/quant_kernel.cu:15-103): per-token absmax quantisation,
 * scale[m] = absmax/127, q = int8(nearbyint(x * (127/absmax))).  x (M,K) f16/bf16 row stride ldx; q (M,K) int8. */
int zl_int8_quant_per_token(const void* x, int ldx, void* q, float* scale, int M, int K, int dtype, int pdl,
                            zl_stream_t stream);
/* int8_op::layernorm_quant (quant_kernel.cu:106-227): y = RMSNorm(x)*w/scale in T plus the int8 twin q with
 * qscale[t] = absmax(x*w) * rsqrt / 127. */
int zl_rmsnorm_quant(const void* x, const void* weight, void* y, void* q, float* qscale, int T, int D, float eps,
                     float scale, int dtype, int pdl, zl_stream_t stream);
/* nn::fp8::dynamic_scaled_quant (src/nn/quant/fp8/fp8_util.cu:110-228): *scale = absmax/448 over all n elements,
 * q = e4m3(sat(x * (1/scale))) with the reference's fp16 product rounding.  n <= 4 Mi elements (decode sizes). */
int zl_fp8_quant_per_tensor(const void* x, void* q, float* scale, size_t n, int dtype, int pdl, zl_stream_t stream);
/* Int8Linear::forward GEMM + int8_op::quant_scale_back (+add_bias), or Fp8Linear::forward's scaled fp8 GEMM, as ONE
 * kernel: y(M,N) = T(acc * x_scale * w_scale) (+bias).  xq (M,K) int8/e4m3; w (N,K) int8/e4m3 row-major (the
 * reference's parameter layout); kind ZL_W8_INT8: x_scale (M) f32, w_scale (N) of w_scale_dtype (ZL_F32 or dtype);
 * kind ZL_W8_FP8: both scales one f32.  INT8 results are bit-identical to the reference's three-kernel path. */
/* int8_op::quant_scale_back (quant_kernel.cu:231-306) stand-alone: y = T(float(acc) * x_scale[m] * w_scale[n]). */
int zl_int8_scale_back(const int32_t* acc, const float* x_scale, const void* w_scale, int w_scale_dtype, void* y, int M,
                       int N, int dtype, zl_stream_t stream);
int zl_w8a8_gemm(const void* xq, const float* x_scale, const void* w, const void* w_scale, int w_scale_dtype,
                 const void* bias, void* y, int M, int N, int K, int kind, int dtype, int pdl, zl_stream_t stream);

/* functions::Gemm / NormalLinear for skinny M (lm_head, bf16 models; src/nn/linear/linear.cpp:150-430,
 * src/nn/embedding/embedding.cu:353-392): y(M,N) = x(M,K) @ W(N,K)^T (+bias), dtype f16/bf16,
 * out_dtype f16/bf16/f32. */
int zl_dense_gemm_skinny(const void* x, int ldx, const void* w, const void* bias, void* y, int M, int N, int K,
                         int dtype, int out_dtype, int pdl, zl_stream_t stream);

/* ------------------------------------------------------------------------------------------ *
 * Norm / residual / activation
 * ------------------------------------------------------------------------------------------ */
/* nn::LayerNorm::forward, rms (src/nn/layernorm/layernorm.cu:9-42): y = T(x*rsqrt(mean(x^2)+eps)*w/scale). */
int zl_rmsnorm(const void* x, const void* weight, void* y, int T, int D, float eps, float scale, int dtype,
               int pdl, zl_stream_t stream);
/* Residual + RMSNorm.  mode 0: block.cpp:124-131 order -- out_sum = T(a+b) (block_kernel.cu:7-17),
 * y = rmsnorm(out_sum);  mode 1: LayerNorm::fuse_add (layernorm.cu:28-41) -- y normalises the unrounded sum.
 * b may be NULL (then out_sum = a).  out_sum may alias a. */
int zl_add_rmsnorm(const void* a, const void* b, const void* weight, void* out_sum, void* y, int T, int D,
                   float eps, float scale, int mode, int dtype, int pdl, zl_stream_t stream);
/* nn::element_add_scale (src/nn/block/block_kernel.cu:7-17), scale_residual=false:
 * c = T(a + T(b*scale))  computed in T. */
int zl_element_add_scale(const void* a, const void* b, void* c, size_t n, float scale, int dtype,
                         zl_stream_t stream);
/* nn::gate_mul_inplace (src/nn/linear/activation_kernel.cu:55-106): out = T(act(float(gate))*float(up));
 * act 0 = silu, 1 = gelu.  gate/up (T, F) with row strides.  up == NULL: out = T(act(gate)), the activation
 * Linear::activate applies (src/nn/linear/linear.cpp activate(), activation_kernel.cu). */
int zl_gate_mul(const void* gate, int ld_gate, const void* up, int ld_up, void* out, int ld_out, int T, int F,
                int act, int dtype, zl_stream_t stream);

/* ------------------------------------------------------------------------------------------ *
 * RoPE + KV append
 * ------------------------------------------------------------------------------------------ */
/* RopePreparer (src/nn/position/rope_preparer.cu:49-161): cos/sin fp32 (T, d).
 * llama3_factor <= 0 -> plain rope. */
int zl_rope_cos_sin(const int32_t* pos, float* cos_out, float* sin_out, int T, int dim_head, float theta,
                    float llama3_factor, float low_freq_factor, float high_freq_factor, float old_context_len,
                    int neox, zl_stream_t stream);
/* nn::rope_qk_cache (src/nn/position/rotary_embedding_fuse_cache.cu:23-125): split fused qkv and rotate q,k. */
int zl_rope_qk_cache(const float* cos, const float* sin, const void* qkv, void* q, void* k, void* v, int T,
                     int num_heads, int num_kv_heads, int dim_head, int neox, int dtype, zl_stream_t stream);
/* nn copy_to_rag_buffer2 (src/kvcache/ragged_buffer_kernel.cu:194-300). */
int zl_copy_to_rag_buffer2(const int32_t* placement, const int32_t* buf_lens, const void* k_src,
                           const void* v_src, void* const* k_addrs, void* const* v_addrs, int B, int len_q,
                           int num_kv_heads, int dim_head, int bshd, int dtype, zl_stream_t stream);
/* Fused: split qkv (+bias already applied) + RoPE(q,k) + append K/V rows at placement into the per-task
 * buffers + write rotated q.  Replaces rope_qk_cache + copy_to_rag_buffer2 (attention.cpp:865-898, 636-676).
 * token_batch (T) int32: task index of each token; placement (T) int32 (<0: skip append). */
int zl_qkv_rope_append(const float* cos, const float* sin, const void* qkv, void* q_out,
                       const int32_t* token_batch, const int32_t* placement, void* const* k_addrs,
                       void* const* v_addrs, int T, int num_heads, int num_kv_heads, int dim_head, int neox,
                       int bshd, const int32_t* buf_lens, int dtype, int pdl, zl_stream_t stream);

/* ------------------------------------------------------------------------------------------ *
 * Decode attention over per-task ragged KV buffers
 * nn::multi_query_attention_rag_buffer (src/nn/attention/attention_kernel.cu:1252-1457)
 * ------------------------------------------------------------------------------------------ */
/* one-shot hint: the NEXT zl_decode_attention call on this thread also prefetches [ptr, ptr+bytes) into L2
 * (weights of a later GEMM; attention leaves HBM idle at small batch). */
int zl_decode_attention_set_prefetch(const void* ptr, size_t bytes);
size_t zl_decode_attention_workspace_bytes(int B, int len_q, int num_heads, int dim_head, int max_len_buf);
/* tests: host view of the launch zl_decode_attention makes for this shape (the same code chooses it): *kernel = 0
 * k_decode_attn (P.V on the tensor cores), 1 warp-per-32-keys kernel, 2 / 3 the ZL_ATTN_OLD_SHORT / ZL_ATTN_PV_FP32
 * variants; *splits = KV splits, each CTA covering round16(ceil(len_buf / splits)) keys of its task. */
int zl_decode_attention_plan(int B, int len_q, int num_heads, int num_kv_heads, int max_len_buf, int* kernel,
                             int* splits);
/* q (B, len_q, H_q, d); buf_lens (B); k_addrs/v_addrs (B) device arrays of device pointers;
 * mask int8 ragged concat of (len_q, len_buf_b); out (B, len_q, H_q, d).  bshd: (len_buf, H_kv, d) else
 * (H_kv, len_buf, d). */
int zl_decode_attention(const void* q, const int32_t* buf_lens, void* const* k_addrs, void* const* v_addrs,
                        const int8_t* mask, float scale, int max_len_buf, void* out, int B, int len_q,
                        int num_heads, int num_kv_heads, int dim_head, int bshd, void* workspace,
                        size_t workspace_bytes, int dtype, int pdl, zl_stream_t stream);

/* int8 KV cache (KV_CACHE_DTYPE=int8 of the reference): KERNEL_mqa_rag_buffer_split_kv_quant
 * (src/nn/attention/attention_kernel.cu:804-880, src/nn/attention/quant_attention.cuh:10-123).  K / V buffers per task are
 * (len_buf, H_kv, d) uint8 = round(x * 127 / absmax) + 128, scale buffers (len_buf, H_kv) fp32 = absmax / 127 (BSHD only,
 * like the reference); q is fp16; out in out_dtype.  Any max_len_buf (the reference only takes this path above
 * ATTN_SPLIT_KV_THRES = 1024).  workspace as zl_decode_attention_workspace_bytes. */
int zl_decode_attention_kv8(const void* q, const int32_t* buf_lens, void* const* k_addrs, void* const* v_addrs,
                            void* const* scale_k_addrs, void* const* scale_v_addrs, const int8_t* mask, float scale,
                            int max_len_buf, void* out, int B, int len_q, int num_heads, int num_kv_heads, int dim_head,
                            void* workspace, size_t workspace_bytes, int out_dtype, int pdl, zl_stream_t stream);
/* cache side of the same contract: int8_op::quant_calc_scale(x, 127, 128) per (token, kv head) row
 * (src/nn/quant/int8/quant_kernel.cu:15-47) + copy_to_rag_buffer2 of the codes and of the scales
 * (src/nn/attention/attention.cpp:656-676): k_src / v_src (T, H_kv, d), token t goes to row placement[t] of task
 * token_batch[t] (placement < 0: skipped). */
/* the same quantisation on dense rows: x (M, K) -> q (M, K) uint8, scale (M) fp32 (quant_calc_scale(x, 127, 128)). */
int zl_int8_quant_rows_u8(const void* x, void* q, float* scale, int M, int K, int dtype, zl_stream_t stream);
int zl_kv_int8_quant_append(const void* k_src, const void* v_src, const int32_t* token_batch, const int32_t* placement,
                            void* const* k_addrs, void* const* v_addrs, void* const* scale_k_addrs,
                            void* const* scale_v_addrs, int T, int num_kv_heads, int dim_head, int dtype, int pdl,
                            zl_stream_t stream);

/* ------------------------------------------------------------------------------------------ *
 * Decode-step helpers around the layers
 * ------------------------------------------------------------------------------------------ */
/* nn::Embedding lookup (src/nn/embedding/embedding.cu:20-60): out[t,:] = table[ids[t],:]. */
int zl_embedding(const int32_t* ids, const void* table, void* out, int T, int D, int vocab, int dtype, int pdl,
                 zl_stream_t stream);
/* greedy pick (generator/batch_generator.cpp:1762-1884 with beam 1): argmax over fp32 logits (T, V). */
size_t zl_argmax_workspace_bytes(int T);
int zl_argmax(const float* logits, int32_t* out, int T, int V, void* workspace, size_t workspace_bytes, int pdl,
              zl_stream_t stream);
/* vocab-parallel pick: per-token {float value, int global index} candidate of one logits shard (T, V), and the
 * merge over the all-gathered candidates [ranks][stride] (embedding.cu:353-392 gathers the logits instead). */
int zl_argmax_candidates(const float* logits, void* cand_out, int T, int V, int idx_offset, void* workspace,
                         size_t workspace_bytes, int pdl, zl_stream_t stream);
int zl_argmax_merge(const void* cand_all, int32_t* out, int T, int ranks, int stride, int pdl, zl_stream_t stream);
/* Seeded sampling pick over fp32 logits (T, V), one launch for all rows.  Row b belongs to task row_task[b] (device
 * int32, each task at most once per call) whose parameters are params[task] (device array):
 *   penalties on every token t set in the task's seen bits (uint32[ceil(V/32)] per task), beam_util.cu:198-220:
 *     presence_penalty != 0 ? l[t] -= presence_penalty : l[t] = l[t] < 0 ? l[t] * rep : l[t] / rep;
 *   random iff top_p < 1 || top_k > 0 (batch_generator.h:106); otherwise the argmax of the penalised logits (ties ->
 *     lowest index, as zl_argmax); defaults (rep 1, presence 0, top_p 1, top_k 0) are plain greedy;
 *   p = softmax(l / temperature) (softmax.cu:10-30), cum = inclusive sum of p sorted descending (ties in ascending
 *     index order), P = top_k > 0 ? min(top_p, cum[top_k-1]) : top_p, v = u * P * cum[V-1], pick the first sorted
 *     position with cum >= v (random_util.cu:83-106);
 *   u = zl_sample_uniform(seed, draw_counters[task]).
 * Then sets the pick's seen bit, advances draw_counters[task] and writes out[b].  The logits are not modified.
 * Requires temperature > 0, 0 <= top_p <= 1, 0 <= top_k < V (random_util.cu:121-122; checked by
 * zl_llama_set_sampling, not here).  Computes in fp32 / fp64 on the fp32 logits; V <= 327680. */
typedef struct zl_sample_params {
    float temperature, top_p, repetition_penalty, presence_penalty;
    int top_k;
    uint64_t seed;
} zl_sample_params_t;
size_t zl_sample_workspace_bytes(int T, int V);
int zl_sample(const float* logits, int T, int V, const int32_t* row_task, const zl_sample_params_t* params,
              uint32_t* seen_bits, uint32_t* draw_counters, int32_t* out, void* workspace, size_t workspace_bytes,
              int pdl, zl_stream_t stream);
/* host: the u in (0, 1] the kernel draws: Philox4x32-10 with key = seed, counter = {draw_index, 0, 0, 0},
 * u = ((w0 >> 8) + 1) * 2^-24.  (The reference draws with curand; the stream differs, the distribution does not.) */
float zl_sample_uniform(uint64_t seed, uint64_t draw_index);
/* synthetic-checkpoint generators (bench / tests): counter-based hash RNG, reproducible per seed. */
int zl_fill_random_u32(uint32_t* p, size_t n, uint64_t seed, zl_stream_t stream);
int zl_fill_const_u32(uint32_t* p, size_t n, uint32_t value, zl_stream_t stream);
int zl_fill_uniform(void* p, size_t n, float lo, float hi, uint64_t seed, int dtype, zl_stream_t stream);

/* ------------------------------------------------------------------------------------------ *
 * Tensor-parallel exchange over NVLink peer memory (one process per GPU, one node)
 * Replaces ModelContext::reduce_sum / reduce_sum2 / reduce_tp_int8 (src/model/model_context.cpp:203-326) and
 * the c10d NCCL wrappers it calls (3rd/bmengine/bmengine/c10d/c10d.cpp:42-136) on the decode path.
 * ------------------------------------------------------------------------------------------ */
/* Allocates this rank's symmetric buffer (inboxes for world_size sources x 2 parities of max_elems 16-bit values). */
int zl_comm_create(int rank, int world_size, size_t max_elems_16bit, zl_comm_t** out);
void zl_comm_destroy(zl_comm_t* c);
int zl_comm_rank(zl_comm_t* c);
int zl_comm_world_size(zl_comm_t* c);
/* CUDA IPC handle of the symmetric buffer (zl_comm_ipc_handle_bytes() bytes); exchange them out of band
 * (torch.distributed all_gather in zhilight_b200/dist.py) and hand all of them (index = rank) to open_peers. */
int zl_comm_ipc_handle_bytes(void);
int zl_comm_get_ipc_handle(zl_comm_t* c, void* handle_out);
int zl_comm_open_peers(zl_comm_t* c, const void* handles_all);
/* once per decode step that uses the exchange fused into the W4 GEMMs (tp_mode of zl_w4a16_gemm_fused), before the first
 * such GEMM of the step and on every rank: advances the step counter the word tags are derived from. */
int zl_comm_ll_begin_step(zl_comm_t* c, zl_stream_t stream);
/* out = T(T(sum over ranks of partial) + residual); n % 32 == 0; residual may be NULL; out may alias residual.
 * int8_payload != 0: peers' contributions travel as int8 + one T scale per 32 values (the reference's group-32
 * format, int8/quant_reduce_kernel.cu:14-38); deterministic rank-ordered fp32 reduction either way. */
int zl_allreduce_one_shot(zl_comm_t* c, const void* partial, const void* residual, void* out, size_t n, int dtype,
                          int int8_payload, int pdl, zl_stream_t stream);
/* out[r*bytes ..] = `in` of rank r (bytes % 16 == 0, small: one CTA). */
int zl_allgather_small(zl_comm_t* c, const void* in, void* out, size_t bytes, int pdl, zl_stream_t stream);
/* int8_op::quant_group_32 / dequant_sum_quant_g32 / dequant_group_32 / dequant_group_fuse_add
 * (src/nn/quant/int8/quant_reduce_kernel.cu:14-38, 243-322, 105-140, 201-240); M = number of 32-groups. */
int zl_quant_group_32(const void* in, int8_t* out_q, void* out_scale, size_t M, int dtype, zl_stream_t stream);
int zl_dequant_sum_quant_g32(const void* my, const int8_t* q_others, const void* scale_others, int8_t* out_q,
                             void* out_scale, size_t M, int world_size, int dtype, zl_stream_t stream);
/* add != NULL: dequant_group_fuse_add (out = q*s + add). */
int zl_dequant_group_32(const int8_t* q, const void* scale, const void* add, void* out, size_t M, int dtype,
                        zl_stream_t stream);

/* ------------------------------------------------------------------------------------------ *
 * Decode driver: the model::LLaMA::encode + get_logits + greedy pick stand-in
 * (src/model/llama.cpp:75-165, src/nn/block/block.cpp:86-143, src/nn/attention/attention.cpp:846-964,
 *  src/nn/feedforward/feedforward.cpp:113-137) for len_q = 1 dynamic-batch steps.  The reference keeps
 * its scheduler (src/generator) above this; here the caller supplies (token, position) per task.
 * One CUDA graph per batch size, all kernels chained with programmatic dependent launch.
 * ------------------------------------------------------------------------------------------ */
typedef struct zl_llama zl_llama_t;
typedef struct zl_llama_config {
    int num_layers, dim_model, num_heads, num_kv_heads, dim_head, dim_ff, vocab_size;
    float eps, rope_theta;
    float rope_llama3_factor; /* <= 0: plain rope */
    float rope_low_freq_factor, rope_high_freq_factor, rope_orig_ctx;
    int quant_type; /* model_config.hpp:132-144 QuantType: 0 none, 2 AutoInt8 (fp weights quantised per row at load),
                     * 5 GPTQ, 6 AWQ, 7 FP8 (e4m3 weights + per-tensor weight_scale), 8 GPTQ_Marlin (= 5 with sym) */
    int group_size, sym;
    int dtype; /* ZL_F16 / ZL_BF16 (W4 paths are fp16-only like the reference, q_gemm_k_major.cu:989) */
    int max_batch, max_seq;
    int tp_rank, tp_size;
    int use_pdl, use_graph;
    int tp_int8; /* TP all-reduce payload: 0 = activation dtype, 1 = int8 group-32 (REDUCE_TP_INT8 of the reference) */
    int fuse; /* 0: one kernel per reference operator; 1: RMSNorm folded into the W4 GEMMs; 2 (3 is accepted as 2):
               * + qkv RoPE/KV-append epilogue.  Launches with more than 16 tokens run zl_rmsnorm + the tcgen05 GEMM. */
    int prefill_chunk; /* 0: decode only.  1..2048: zl_llama_prefill processes a prompt in chunks of this many tokens
                        * (chunked prefill, zhilight/config/adapter.py:47-48) */
    int qkv_bias; /* zl_llama_init_synthetic: also create q/k/v biases (Qwen2: attention.cpp:105-109); loaded checkpoints
                   * carry their ".bias" tensors regardless of this flag */
} zl_llama_config_t;

int zl_llama_create(const zl_llama_config_t* cfg, zl_llama_t** out);
/* tensor parallel: hand the driver its exchange object (zl_comm_create + open_peers) before the first step. */
int zl_llama_set_comm(zl_llama_t* m, zl_comm_t* comm);
void zl_llama_destroy(zl_llama_t* m);
/* Stage one checkpoint tensor (HOST pointer, row-major (rows, cols)); names as produced by
 * zhilight/loader.py:250-358 without the "llama." prefix, e.g. "layers.0.attn.project_q.qweight". */
int zl_llama_load_tensor(zl_llama_t* m, const char* name, const void* data_host, int rows, int cols,
                         int elem_bytes);
/* Fill every tensor of the configured architecture with reproducible random data ON DEVICE
 * (HF-GPTQ layout for quantized linears) and run the load pipeline layer by layer. */
int zl_llama_init_synthetic(zl_llama_t* m, uint64_t seed);
/* Run the load pipeline (Int4GPTQ::preprocess_weight + fusion + ZLW4 pack) on the staged tensors. */
int zl_llama_finalize(zl_llama_t* m);
/* One decode step for B tasks.  tokens_host/positions_host (B) int32; task b owns KV slot b.
 * next_tokens_host (B) int32 greedy picks; logits_host NULL or (B, vocab) fp32.  Synchronous. */
int zl_llama_decode(zl_llama_t* m, const int32_t* tokens_host, const int32_t* positions_host, int B,
                    int32_t* next_tokens_host, float* logits_host);
/* Device-resident variant: stage tokens/positions once, then each call replays the step, feeds the picked
 * tokens back and advances positions on the device; no host sync. */
int zl_llama_set_state(zl_llama_t* m, const int32_t* tokens_host, const int32_t* positions_host, int B);
int zl_llama_step_device(zl_llama_t* m, int B);
/* read back the device-resident (token, position) state; synchronous. */
int zl_llama_get_state(zl_llama_t* m, int32_t* tokens_host, int32_t* positions_host, int B);
/* read back the fp32 logits (B, vocab/tp) of the most recent decode step (this rank's shard); synchronous. */
int zl_llama_get_logits(zl_llama_t* m, float* logits_host, int B);
int zl_llama_sync(zl_llama_t* m);
/* Chunked prefill of ONE task (SearchTask prompt, src/generator/batch_generator.cpp:1576): appends tokens_host[0..n) at
 * positions pos0.. to the task's KV buffers through the same kernels (M = chunk GEMMs, causal len_q = chunk attention)
 * and returns the greedy next token (and optionally the last position's logits, vocab/tp floats).  Synchronous. */
/* Prefill keeps its own token / position staging on the device: the (token, position) state of the decode tasks set by
 * zl_llama_set_state survives a prefill issued between two zl_llama_step_device calls (continuous batching).  It
 * overwrites the next-token / logits row 0 outputs, which zl_llama_step_device consumes before it returns. */
int zl_llama_prefill(zl_llama_t* m, int task, const int32_t* tokens_host, int n, int pos0, int32_t* next_token_host,
                     float* logits_host);
/* Sampling state of one task (SearchTask's temperature / top_p / top_k / repetition_penalty / presence_penalty /
 * seed, batch_generator.cpp:1639-1692): validates host_params, copies them to the device and clears the task's seen
 * set and draw counter.  Steps whose batch holds a task with such state pick with zl_sample instead of zl_argmax (a
 * graph of its own; later parameter changes reuse it).  tp_size > 1: ZL_ERR_UNSUPPORTED (top-p over vocabulary shards
 * needs a global select). */
int zl_llama_set_sampling(zl_llama_t* m, int task, const zl_sample_params_t* host_params);
/* back to plain greedy picks for this task. */
int zl_llama_clear_sampling(zl_llama_t* m, int task);
zl_stream_t zl_llama_stream(zl_llama_t* m);
/* bytes the step must read from HBM per rank (weights + lm_head + norms), kernel launches per step. */
int zl_llama_stats(zl_llama_t* m, int B, double* weight_bytes, int* kernels_per_step);
/* Roofline probe for the dominant kernel: enqueue only the W4A16 (or dense) GEMMs of one decode step
 * (every layer's own weights, same PDL chain) `iters` times between CUDA events on the driver's stream.
 * Returns total milliseconds, the number of GEMM launches and their algorithmic bytes. */
int zl_llama_bench_gemms(zl_llama_t* m, int B, int iters, float* ms, int* launches, double* bytes);

#ifdef __cplusplus
}
#endif
#endif /* ZHILIGHT_B200_H_ */
