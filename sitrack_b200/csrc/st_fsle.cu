// st_fsle.cu -- finite-size Lyapunov exponents (FSLE) of buoy pairs: per-pair first-passage state kept on the device
// across the whole run, and per-sample statistics of the exit times between separation thresholds (Aurell et al.
// 1997; Lacorata et al. 2001; LaCasce 2008).
//
// Definitions (DESIGN.md section 14, oracle/fsle_ref.py).  Per pair (a, b) and sample t, in f8 and in this order:
//   dy = y_a - y_b, dx = x_a - x_b, r = sqrt(dy*dy + dx*dx);  valid when both masks != 0 and r is finite;
//   b = bin_right(deltas, K, r), the number of thresholds at or below r.
// State int2 {level, anchor}: level -1 not started, -2 ended, 0..K thresholds reached; anchor the sample at which the
// level was first reached, -1 when unknown.  Not started and valid: level = b, anchor = -1, n_start[b]++.  Started and
// not valid: ended; censored[level-1]++ when anchor >= 0 and level < K.  Started, valid and b > level: tau = t - anchor
// for transition level-1 (if level >= 1 and anchor >= 0), tau = 0 for transitions level .. b-2, then anchor = t and
// level = b.  Each recorded tau adds 1 to hist_tau[j][bin_right(tau_edges, tau)], tau to sum_tau[j] and tau^2 to
// sum_tau2[j].  Every output is an integer: shared-memory counters (32-bit counts, 64-bit sums) flushed with integer
// atomics, so the statistics are exact and do not depend on the launch grid, the device or the buoy storage order.
//
// Kernel, on the caller's stream: k_fsle, one thread per pair, grid-strided over blocks of FS_BLOCK pairs.
#include "st_deform.cuh"

namespace st {

constexpr int FS_BLOCK = 256;

// shared memory: deltas (K f8), tau_edges (ntau f8), sum_tau and sum_tau2 ((K-1) u64 each), then the 32-bit counters
// n_start (K+1), hist_tau ((K-1)(ntau+1)) and n_censored (K-1)
size_t fsle_smem(int K, int ntau)
{
    const size_t J = (size_t)K - 1;
    return ((size_t)K + ntau + 2 * J) * 8 + ((size_t)K + 1 + J * (ntau + 1) + J) * 4;
}

long long fsle_stats_len(int K, int ntau)
{
    return (long long)(K + 1) + (long long)(K - 1) * (ntau + 1) + 3LL * (K - 1);
}

struct FsleCounters {
    const double* de;
    const double* te;
    unsigned long long* sum;           // sum_tau [K-1], then sum_tau2 [K-1]
    int* nst;                          // n_start [K+1]
    int* hist;                         // hist_tau [K-1][ntau+1]
    int* cens;                         // n_censored [K-1]
    int K, ntau;

    __device__ __forceinline__ void record(int j, int tau) const
    {
        atomicAdd(hist + j * (ntau + 1) + bin_right(te, ntau, (double)tau), 1);
        if (tau) {
            atomicAdd(sum + j, (unsigned long long)tau);
            atomicAdd(sum + (K - 1) + j, (unsigned long long)tau * (unsigned long long)tau);
        }
    }

    // one sample t of one pair: (level, anchor) updated in place
    __device__ __forceinline__ void update(int& level, int& anchor, bool mok, pt pa, pt pb, int t) const
    {
        const double dy = __dsub_rn(pa.y, pb.y), dx = __dsub_rn(pa.x, pb.x);
        const double r = __dsqrt_rn(__dadd_rn(__dmul_rn(dy, dy), __dmul_rn(dx, dx)));
        const bool valid = mok && isfinite(r);
        if (level == -1) {
            if (valid) {
                level = bin_right(de, K, r);
                anchor = -1;
                atomicAdd(nst + level, 1);
            }
        } else if (!valid) {
            if (anchor >= 0 && level < K) atomicAdd(cens + level - 1, 1);
            level = -2;
        } else {
            const int b = bin_right(de, K, r);
            if (b > level) {
                if (level >= 1 && anchor >= 0) record(level - 1, t - anchor);
                for (int j = level; j <= b - 2; ++j) record(j, 0);
                anchor = t;
                level = b;
            }
        }
    }
};

__global__ void __launch_bounds__(FS_BLOCK) k_fsle(long long nQ, const int2* __restrict__ pairs, int2* __restrict__ state,
                                                   const pt* __restrict__ yx, const int8_t* __restrict__ m, int t,
                                                   const pt* __restrict__ yx0, const int8_t* __restrict__ m0, int K,
                                                   const double* __restrict__ deltas, int ntau,
                                                   const double* __restrict__ tau_edges,
                                                   unsigned long long* __restrict__ stats)
{
    extern __shared__ double s_dyn[];
    const int J = K - 1, nhist = J * (ntau + 1);
    FsleCounters c;
    c.K = K; c.ntau = ntau;
    double* de = s_dyn;
    double* te = de + K;
    c.de = de; c.te = te;
    c.sum = reinterpret_cast<unsigned long long*>(te + ntau);
    c.nst = reinterpret_cast<int*>(c.sum + 2 * J);
    c.hist = c.nst + K + 1;
    c.cens = c.hist + nhist;
    for (int k = threadIdx.x; k < K; k += FS_BLOCK) de[k] = deltas[k];
    for (int k = threadIdx.x; k < ntau; k += FS_BLOCK) te[k] = tau_edges[k];
    for (int k = threadIdx.x; k < 2 * J; k += FS_BLOCK) c.sum[k] = 0ull;
    for (int k = threadIdx.x; k < K + 1 + nhist + J; k += FS_BLOCK) c.nst[k] = 0;
    __syncthreads();
    for (long long i = (long long)blockIdx.x * FS_BLOCK + threadIdx.x; i < nQ; i += (long long)gridDim.x * FS_BLOCK) {
        const int2 q = __ldcs(pairs + i);
        int2 s0 = yx0 ? make_int2(-1, -1) : __ldcs(state + i);       // a start row resets the pair
        if (s0.x == -2) continue;                                      // ended: no gathers
        int level = s0.x, anchor = s0.y;
        if (yx0) {
            // the start row's and the sample row's gathers, issued together
            const int8_t ka0 = __ldg(m0 + q.x), kb0 = __ldg(m0 + q.y), ka = __ldg(m + q.x), kb = __ldg(m + q.y);
            const pt pa0 = ld_ro_pt(yx0, q.x), pb0 = ld_ro_pt(yx0, q.y), pa = ld_ro_pt(yx, q.x), pb = ld_ro_pt(yx, q.y);
            c.update(level, anchor, ka0 != 0 && kb0 != 0, pa0, pb0, t - 1);
            c.update(level, anchor, ka != 0 && kb != 0, pa, pb, t);
            __stcs(state + i, make_int2(level, anchor));
        } else {
            const int8_t ka = __ldg(m + q.x), kb = __ldg(m + q.y);
            const pt pa = ld_ro_pt(yx, q.x), pb = ld_ro_pt(yx, q.y);
            c.update(level, anchor, ka != 0 && kb != 0, pa, pb, t);
            if (level != s0.x || anchor != s0.y) __stcs(state + i, make_int2(level, anchor));
        }
    }
    __syncthreads();
    // flush: stats = n_start (K+1), hist_tau (K-1)(ntau+1), sum_tau, sum_tau2, n_censored (K-1 each)
    for (int k = threadIdx.x; k < K + 1 + nhist; k += FS_BLOCK)
        if (c.nst[k]) atomicAdd(stats + k, (unsigned long long)c.nst[k]);
    for (int k = threadIdx.x; k < 2 * J; k += FS_BLOCK)
        if (c.sum[k]) atomicAdd(stats + K + 1 + nhist + k, c.sum[k]);
    for (int k = threadIdx.x; k < J; k += FS_BLOCK)
        if (c.cens[k]) atomicAdd(stats + K + 1 + nhist + 2 * J + k, (unsigned long long)c.cens[k]);
}

cudaError_t launch_fsle(long long nQ, const int32_t* pairs, int32_t* state, const pt* yx, const int8_t* m, int t,
                        const pt* yx0, const int8_t* m0, int K, const double* deltas, int ntau,
                        const double* tau_edges, int64_t* stats, cudaStream_t st)
{
    cudaError_t e = cudaMemsetAsync(stats, 0, sizeof(int64_t) * (size_t)fsle_stats_len(K, ntau), st);
    if (e != cudaSuccess) return e;
    const size_t smem = fsle_smem(K, ntau);
    if (smem > 48 * 1024 &&
        (e = cudaFuncSetAttribute(k_fsle, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess)
        return e;
    // one wave of resident blocks (the statistics are integers: the grid does not change them)
    int dev = 0, nsm = 0, per_sm = 0;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess ||
        (e = cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess ||
        (e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_fsle, FS_BLOCK, smem)) != cudaSuccess)
        return e;
    const long long tiles = (nQ + FS_BLOCK - 1) / FS_BLOCK, wave = (long long)nsm * (per_sm < 1 ? 1 : per_sm);
    const int grid = (int)(tiles < wave ? tiles : wave);
    k_fsle<<<grid, FS_BLOCK, smem, st>>>(nQ, reinterpret_cast<const int2*>(pairs), reinterpret_cast<int2*>(state), yx,
                                         m, t, yx0, m0, K, deltas, ntau, tau_edges,
                                         reinterpret_cast<unsigned long long*>(stats));
    return cudaGetLastError();
}

}  // namespace st
