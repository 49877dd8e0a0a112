// Seeded top-k / top-p sampling with repetition and presence penalties over fp32 logits, one launch for all rows.
//
// Contract (per row b, task = row_task[b], logits row l of length V), following the reference:
//   penalties   (generator/beam_util.cu:198-220) on every token t of the task's seen set:
//               presence != 0 ? l[t] -= presence : l[t] = l[t] < 0 ? l[t] * rep : l[t] / rep;
//   random iff top_p < 1 || top_k > 0 (generator/batch_generator.h:106); otherwise argmax of the penalised logits
//               (ties -> lowest index, as zl_argmax);
//   p = softmax(l / temperature) (functions/softmax.cu:10-30); cum = inclusive sum of p in descending order, ties in
//               ascending index order; P = top_k > 0 ? min(top_p, cum[top_k-1]) : top_p; v = u * P * cum[V-1]; pick the
//               first sorted position with cum >= v (generator/random_util.cu:83-106);
//   u from Philox4x32-10 (philox.h), key = seed, counter = {draw_index, 0, 0, 0}.
// The penalised logits are not written back: the caller's logits stay the raw lm_head output.
//
// No sort.  The pick is a rank / mass select over the composite key (order-preserving descending key of l'/T, index),
// found by radix passes of 4 bits: each pass counts the candidates and sums their exp-mass per digit in registers
// (no shared-memory atomics), the eight CTAs of a thread-block cluster merge their bins through distributed shared
// memory, and the bin holding the target becomes the new candidate prefix.  Once at most kBrute candidates remain,
// every CTA pulls them and ranks them by direct comparison.  Each CTA keeps its slice of l'/T in shared memory, so
// the logits are read from L2 once.
#include "common.cuh"
#include "philox.h"

#include <cooperative_groups.h>

namespace cg = cooperative_groups;

namespace zl {
namespace {

constexpr int kCluster = 8;          // CTAs per row
constexpr int kThreads = 512;
constexpr int kWarps = kThreads / 32;
constexpr int kBins = 16;            // 4-bit digit per pass
constexpr int kBrute = 1024;         // candidates ranked by direct comparison
constexpr int kMaxSlice = 40960;     // floats of l'/T per CTA in dynamic shared memory -> V <= kCluster * kMaxSlice

struct SampleSmem {
    double xmass[2][kBins];          // this CTA's cumulative digit masses / counts, published to the cluster
    unsigned xcnt[2][kBins];
    double tmass[kBins];             // cluster totals of the current pass
    unsigned tcnt[kBins];
    double wmass[kWarps][kBins];     // per-warp partials
    unsigned wcnt[kWarps][kBins];
    float pub_val;                   // phase 0: this CTA's argmax of l' and max of l'/T
    int pub_idx;
    float pub_xmax;
    float red_val[kWarps];
    int red_idx[kWarps];
    float red_x[kWarps];
    unsigned n_local;                // candidates gathered from this CTA's slice
    unsigned n_all;
    unsigned long long best;
    double win_cum;
    unsigned long long lkey[kBrute];
    float le[kBrute];
    unsigned long long akey[kBrute];
    float ae[kBrute];
};

__device__ __forceinline__ uint32_t desc_key(float x) {
    uint32_t b = __float_as_uint(x == 0.0f ? 0.0f : x);            // -0 ranks with +0
    const uint32_t ord = b ^ ((uint32_t)((int32_t)b >> 31) | 0x80000000u);   // ascending with x
    return ~ord;                                                    // ascending key = descending x
}

__device__ __forceinline__ bool better(float v, int i, float bv, int bi) { return v > bv || (v == bv && i < bi); }

struct Select {
    unsigned long long key;   // composite key of the pick
    double cum;               // exp-mass up to and including the pick (descending order)
    double total;             // exp-mass of the whole row
};

// One rank (kind 0: target = rank r) or mass (kind 1: target = u * P * total, P = min(top_p, pcap)) select over the
// whole row.  Called uniformly by every thread of every CTA of the cluster.
__device__ Select cluster_select(SampleSmem& s, const float* xs, int n, int lo, int ib, float xmax, int kind, unsigned r,
                                 double u_p, cg::cluster_group& cl, int& parity) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tot_bits = 32 + ib;
    unsigned long long prefix = 0;
    int shift = tot_bits;          // candidates: composite >> shift == prefix >> shift (all when shift == tot_bits)
    unsigned before_cnt = 0, n_c = 0;
    double before_mass = 0.0, total = 0.0, target = 0.0;
    bool first = true;
    while (first || (n_c > (unsigned)kBrute && shift > 0)) {
        unsigned cnt[kBins];
        float mass[kBins];
#pragma unroll
        for (int b = 0; b < kBins; ++b) {
            cnt[b] = 0;
            mass[b] = 0.f;
        }
        const int dsh = shift - 4;
        for (int j = tid; j < n; j += kThreads) {
            const float x = xs[j];
            const unsigned long long k = ((unsigned long long)desc_key(x) << ib) | (unsigned)(lo + j);
            if (shift < tot_bits && (k >> shift) != (prefix >> shift)) continue;
            const unsigned d = (unsigned)(k >> dsh) & 15u;
            const float e = expf(x - xmax);
#pragma unroll
            for (int b = 0; b < kBins; ++b) {
                const bool in = d <= (unsigned)b;
                cnt[b] += in ? 1u : 0u;
                mass[b] += in ? e : 0.f;
            }
        }
#pragma unroll
        for (int b = 0; b < kBins; ++b) {
            double m = (double)mass[b];
            unsigned c = cnt[b];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                m += __shfl_xor_sync(0xffffffffu, m, o);
                c += __shfl_xor_sync(0xffffffffu, c, o);
            }
            if (lane == 0) {
                s.wmass[warp][b] = m;
                s.wcnt[warp][b] = c;
            }
        }
        __syncthreads();
        if (tid < kBins) {
            double m = 0.0;
            unsigned c = 0;
            for (int w = 0; w < kWarps; ++w) {
                m += s.wmass[w][tid];
                c += s.wcnt[w][tid];
            }
            s.xmass[parity][tid] = m;
            s.xcnt[parity][tid] = c;
        }
        cl.sync();
        if (tid < kBins) {
            double m = 0.0;
            unsigned c = 0;
            for (int q = 0; q < kCluster; ++q) {
                const SampleSmem* rs = cl.map_shared_rank(&s, q);
                m += rs->xmass[parity][tid];
                c += rs->xcnt[parity][tid];
            }
            s.tmass[tid] = m;
            s.tcnt[tid] = c;
        }
        __syncthreads();
        if (first) {
            total = s.tmass[kBins - 1];
            target = kind == 0 ? 0.0 : u_p * total;
        }
        // the bin holding the target (digits ascend with the sorted order)
        int pick = -1, last_nonempty = 0;
        for (int b = 0; b < kBins; ++b) {
            const unsigned cb = s.tcnt[b] - (b ? s.tcnt[b - 1] : 0u);
            if (cb == 0) continue;
            last_nonempty = b;
            if (pick < 0 && (kind == 0 ? before_cnt + s.tcnt[b] > r : before_mass + s.tmass[b] >= target)) pick = b;
        }
        if (pick < 0) pick = last_nonempty;   // rounding left the mass target past the end: the last candidate
        if (pick > 0) {
            before_cnt += s.tcnt[pick - 1];
            before_mass += s.tmass[pick - 1];
        }
        n_c = s.tcnt[pick] - (pick ? s.tcnt[pick - 1] : 0u);
        prefix |= (unsigned long long)pick << dsh;
        shift = dsh;
        parity ^= 1;
        first = false;
    }
    // rank the remaining candidates directly
    if (tid == 0) {
        s.n_local = 0;
        s.best = ~0ull;
    }
    __syncthreads();
    for (int j = tid; j < n; j += kThreads) {
        const float x = xs[j];
        const unsigned long long k = ((unsigned long long)desc_key(x) << ib) | (unsigned)(lo + j);
        if ((k >> shift) != (prefix >> shift)) continue;
        const unsigned slot = atomicAdd(&s.n_local, 1u);
        s.lkey[slot] = k;
        s.le[slot] = expf(x - xmax);
    }
    cl.sync();
    if (warp == 0) {   // pull every CTA's candidates (the total is n_c <= kBrute)
        unsigned off = 0;
        for (int q = 0; q < kCluster; ++q) {
            const SampleSmem* rs = cl.map_shared_rank(&s, q);
            const unsigned nq = rs->n_local;
            for (unsigned i = lane; i < nq; i += 32) {
                s.akey[off + i] = rs->lkey[i];
                s.ae[off + i] = rs->le[i];
            }
            off += nq;
        }
        if (lane == 0) s.n_all = off;
    }
    __syncthreads();
    const unsigned na = s.n_all;
    for (unsigned j = tid; j < na; j += kThreads) {
        const unsigned long long kj = s.akey[j];
        unsigned rank = 0;
        double mb = 0.0;
        for (unsigned c = 0; c < na; ++c) {
            if (s.akey[c] < kj) {
                ++rank;
                mb += (double)s.ae[c];
            }
        }
        const double cum = before_mass + mb + (double)s.ae[j];
        if (kind == 0 ? before_cnt + rank == r : cum >= target) {
            atomicMin(&s.best, kj);
        }
    }
    __syncthreads();
    if (tid == 0 && s.best == ~0ull) {   // no candidate reached the mass target: the last one
        unsigned long long mx = 0;
        for (unsigned j = 0; j < na; ++j) mx = s.akey[j] > mx ? s.akey[j] : mx;
        s.best = mx;
    }
    __syncthreads();
    const unsigned long long win = s.best;
    for (unsigned j = tid; j < na; j += kThreads) {
        if (s.akey[j] != win) continue;
        double mb = 0.0;
        for (unsigned c = 0; c < na; ++c)
            if (s.akey[c] < win) mb += (double)s.ae[c];
        s.win_cum = before_mass + mb + (double)s.ae[j];
    }
    __syncthreads();
    Select res{win, s.win_cum, total};
    return res;
}

__global__ void __cluster_dims__(kCluster, 1, 1) __launch_bounds__(kThreads, 1)
k_sample(const float* __restrict__ logits, int V, const int32_t* __restrict__ row_task,
         const zl_sample_params_t* __restrict__ params, uint32_t* __restrict__ seen_bits,
         uint32_t* __restrict__ draw_counters, int32_t* __restrict__ out, int ib) {
    extern __shared__ float xs[];
    __shared__ SampleSmem s;
    cg::cluster_group cl = cg::this_cluster();
    pdl_trigger();
    pdl_wait();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int rank = (int)cl.block_rank();
    const int row = blockIdx.y;
    const int task = row_task[row];
    const zl_sample_params_t p = params[task];
    const int words = (V + 31) >> 5;
    uint32_t* seen = seen_bits + (size_t)task * words;
    const uint32_t draw = draw_counters[task];
    const bool random = p.top_p < 1.0f || p.top_k > 0;
    const int per = (V + kCluster - 1) / kCluster;
    const int lo = rank * per;
    const int n = max(0, min(V, lo + per) - lo);
    const float* lrow = logits + (size_t)row * V;

    // phase 0: penalties, argmax of l', l'/T into shared memory and its max
    float bv = -INFINITY, bx = -INFINITY;
    int bi = 0x7fffffff;
    for (int j = tid; j < n; j += kThreads) {
        const int i = lo + j;
        float l = lrow[i];
        if ((seen[i >> 5] >> (i & 31)) & 1u)
            l = p.presence_penalty != 0.0f ? l - p.presence_penalty
                                           : (l < 0.0f ? l * p.repetition_penalty : l / p.repetition_penalty);
        if (better(l, i, bv, bi)) {
            bv = l;
            bi = i;
        }
        if (random) {
            const float x = l / p.temperature;
            xs[j] = x;
            bx = fmaxf(bx, x);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (better(ov, oi, bv, bi)) {
            bv = ov;
            bi = oi;
        }
        bx = fmaxf(bx, __shfl_xor_sync(0xffffffffu, bx, o));
    }
    if (lane == 0) {
        s.red_val[warp] = bv;
        s.red_idx[warp] = bi;
        s.red_x[warp] = bx;
    }
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < kWarps; ++w) {
            if (better(s.red_val[w], s.red_idx[w], bv, bi)) {
                bv = s.red_val[w];
                bi = s.red_idx[w];
            }
            bx = fmaxf(bx, s.red_x[w]);
        }
        s.pub_val = bv;
        s.pub_idx = bi;
        s.pub_xmax = bx;
    }
    cl.sync();
    bv = -INFINITY;
    bi = 0x7fffffff;
    bx = -INFINITY;
    for (int q = 0; q < kCluster; ++q) {
        const SampleSmem* rs = cl.map_shared_rank(&s, q);
        const float qv = rs->pub_val;
        const int qi = rs->pub_idx;
        if (better(qv, qi, bv, bi)) {
            bv = qv;
            bi = qi;
        }
        bx = fmaxf(bx, rs->pub_xmax);
    }
    int pick = bi;
    if (random) {
        int parity = 0;
        double u_p = 0.0;
        double pcap = 1.0;
        if (p.top_k > 0) {
            const Select k = cluster_select(s, xs, n, lo, ib, bx, 0, (unsigned)(p.top_k - 1), 0.0, cl, parity);
            pcap = k.cum / (k.total + 1e-20);
        }
        const double u = (double)sample_uniform(p.seed, draw);
        const double P = p.top_k > 0 ? fmin((double)p.top_p, pcap) : (double)p.top_p;
        u_p = u * P;
        const Select m = cluster_select(s, xs, n, lo, ib, bx, 1, 0u, u_p, cl, parity);
        pick = (int)(m.key & ((1ull << ib) - 1));
    }
    if (rank == 0 && tid == 0) {
        out[row] = pick;
        atomicOr(&seen[pick >> 5], 1u << (pick & 31));
        draw_counters[task] = draw + 1;
    }
    cl.sync();   // no CTA leaves while another may still read its shared memory
}

}  // namespace

cudaError_t prepare_sample() {
    return cudaFuncSetAttribute(k_sample, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSlice * (int)sizeof(float));
}

}  // namespace zl

using namespace zl;

extern "C" size_t zl_sample_workspace_bytes(int T, int V) {
    (void)T;
    (void)V;
    return 0;   // the kernel keeps its state in (distributed) shared memory
}

extern "C" float zl_sample_uniform(uint64_t seed, uint64_t draw_index) {
    return sample_uniform(seed, (uint32_t)draw_index);
}

extern "C" int zl_sample(const float* logits, int T, int V, const int32_t* row_task, const zl_sample_params_t* params,
                         uint32_t* seen_bits, uint32_t* draw_counters, int32_t* out, void* workspace,
                         size_t workspace_bytes, int pdl, zl_stream_t stream) {
    (void)workspace;
    ZL_CHECK_ARG(logits && row_task && params && seen_bits && draw_counters && out && T > 0 && V > 1);
    ZL_CHECK_ARG(workspace_bytes >= zl_sample_workspace_bytes(T, V));
    ZL_CHECK_ARG(T <= 65535);
    ZL_CHECK_SUPPORTED(V <= kCluster * kMaxSlice);
    {   // opt-in shared memory once per device (zl_prepare also does it, outside any capture, for the decode driver)
        static bool prepared[64] = {};
        int dev = 0;
        ZL_CHECK_CUDA(cudaGetDevice(&dev));
        if (dev < 0 || dev >= 64 || !prepared[dev]) {
            ZL_CHECK_CUDA(prepare_sample());
            if (dev >= 0 && dev < 64) prepared[dev] = true;
        }
    }
    int ib = 4;
    while (ib < 32 && ((unsigned)(V - 1) >> ib) != 0) ib += 4;   // index bits of the composite key, whole digits
    const int per = (V + kCluster - 1) / kCluster;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(kCluster, T);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = (size_t)per * sizeof(float);
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    zl_count_launch();
    ZL_CHECK_CUDA(cudaLaunchKernelEx(&cfg, k_sample, logits, V, row_task, params, seen_bits, draw_counters, out, ib));
    return ZL_OK;
}
