// st_connect.cu -- buoy transits between regions: per-buoy connectivity state kept on the device across the whole run,
// and per-sample integer statistics of starts, ends, region-to-region transitions, source-to-region occupancy and
// first-arrival times (DeRepentigny et al. 2016; Newton et al. 2017).
//
// Definitions (DESIGN.md section 16, oracle/connect_ref.py).  A label map labels (Nj*Ni) u8 on the T-grid, regions
// 1..R (R = nreg <= 31), 0 = in no region, a label above R counted as 0.  Per buoy p of sample t: its cell (jT, iT)
// from the cell word (bit 31 stripped), its row mask m; valid when m != 0 and 1 <= jT <= Nj-2, 1 <= iT <= Ni-2;
// cur = labels[jT*Ni + iT] when valid.  State (8 B): word x = visited (bit r-1 for region r), word y = start | src<<16 |
// prev<<21 | status<<26 (status 0 not started, 1 started, 2 ended; all zero = not started).
//   not started, valid:    src = prev = cur, start = t, visited = bit(cur); n_start[src]++, count[src][cur]++ (t > 0);
//   started, not valid:    ended for good; n_end[src]++;
//   started, valid:        trans[prev][cur]++, count[src][cur]++; cur >= 1 not yet visited: a first arrival with
//                          tau = t - start: n_arrive[src][cur-1]++, sum_tau += tau, sum_tau2 += tau^2,
//                          hist_tau[src][cur-1][bin_right(tau_edges, tau)]++, bit set; then prev = cur.
// t = 0 resets every buoy before it is evaluated, and adds no count (sample 0's snapshot is diag(n_start)).
//
// Kernel, on the caller's stream: k_connect, one thread per buoy over one wave of resident blocks, grid-strided by
// warp tiles so that every lane of a warp reaches the warp-wide aggregation below together.  The cell word, the mask
// and the state stream through (touch once, issued together); the label is gathered only for valid buoys that have
// not ended, through the read-only path with the L2 evict_last policy (the map stays resident in L2); the state is
// written back only when it changes.  Counters: n_start, n_end, count, trans, n_arrive as 32-bit and sum_tau, sum_tau2
// as 64-bit words in shared memory, added to once per distinct key of a warp (a uniform key by one shuffle and vote,
// otherwise __match_any_sync) by the lowest lane holding it; flushed where non-zero with 64-bit integer atomics.
// hist_tau (up to 32 x 31 x 513 words) goes warp-aggregated straight to global atomics: its events are first
// arrivals, at most R per buoy and run.  Integers throughout: the statistics do not depend on the launch grid, the
// device, the buoy storage order or the split of the buoys between calls.
#include "st_deform.cuh"

namespace st {

constexpr int CN_BLOCK = 256;
constexpr unsigned CN_FULL = 0xffffffffu;

// 32-bit counter words n_start (R+1), n_end (R+1), count, trans ((R+1)^2 each), n_arrive ((R+1) R); the 64-bit
// sum_tau, sum_tau2 ((R+1) R each) follow them in the statistics buffer, hist_tau ((R+1) R (ntau+1)) last
static __host__ __device__ __forceinline__ long long cn_n32(int R)
{
    return 2LL * (R + 1) + 2LL * (R + 1) * (R + 1) + (long long)(R + 1) * R;
}

size_t connect_smem(int R)
{
    return (size_t)(2LL * (R + 1) * R) * 8 + (size_t)cn_n32(R) * 4;
}

long long connect_stats_len(int R, int ntau)
{
    return cn_n32(R) + 2LL * (R + 1) * R + (long long)(R + 1) * R * (ntau + 1);
}

__device__ __forceinline__ unsigned cn_label(const uint8_t* __restrict__ a, int i)
{
    unsigned r;
    asm("ld.global.nc.L2::cache_hint.u8 %0, [%1], %2;" : "=r"(r) : "l"(a + i), "l"(l2_keep_policy()));
    return r;
}

// peers of this lane's key in the warp (every lane calls it)
__device__ __forceinline__ unsigned cn_peers(int key)
{
    if (__all_sync(CN_FULL, key == __shfl_sync(CN_FULL, key, 0))) return CN_FULL;
    return __match_any_sync(CN_FULL, key);
}

__global__ void __launch_bounds__(CN_BLOCK) k_connect(long long nP, int Nj, int Ni, const uint8_t* __restrict__ labels,
                                                     int R, const int2* __restrict__ cell,
                                                     const int8_t* __restrict__ mask, int t, int2* __restrict__ state,
                                                     int ntau, const double* __restrict__ tau_edges,
                                                     unsigned long long* __restrict__ stats)
{
    extern __shared__ unsigned long long s_cn[];
    const int R1 = R + 1, NB = ntau + 1;
    const int n64 = 2 * R1 * R, n32 = (int)cn_n32(R);
    unsigned long long* s_sum = s_cn;                               // sum_tau [R1][R], then sum_tau2 [R1][R]
    unsigned* s32 = reinterpret_cast<unsigned*>(s_cn + n64);        // n_start | n_end | count | trans | n_arrive
    const int o_end = R1, o_count = 2 * R1, o_trans = 2 * R1 + R1 * R1, o_arr = 2 * R1 + 2 * R1 * R1;
    for (int k = threadIdx.x; k < n64; k += CN_BLOCK) s_sum[k] = 0ull;
    for (int k = threadIdx.x; k < n32; k += CN_BLOCK) s32[k] = 0u;
    __syncthreads();
    unsigned long long* g_hist = stats + n32 + n64;
    const unsigned lane = threadIdx.x & 31u;
    const long long stride = (long long)gridDim.x * CN_BLOCK;
    for (long long p0 = (long long)blockIdx.x * CN_BLOCK + (threadIdx.x & ~31u); p0 < nP; p0 += stride) {
        const long long p = p0 + lane;
        const bool in = p < nP;
        int2 cw = make_int2(0, 0), s = make_int2(0, 0);
        int8_t m = 0;
        if (in) {
            cw = __ldcs(cell + p);
            m = __ldcs(mask + p);
            if (t) s = __ldcs(state + p);                           // t = 0: every buoy starts afresh
        }
        const unsigned w = (unsigned)s.y;
        const unsigned status = (w >> 26) & 3u, src = (w >> 16) & 31u, prev = (w >> 21) & 31u, start = w & 0xffffu;
        const int jT = cw.x & 0x7fffffff, iT = cw.y;
        const bool valid = in && m != 0 && jT >= 1 && jT <= Nj - 2 && iT >= 1 && iT <= Ni - 2;
        unsigned cur = 0;
        if (valid && status != 2u) {
            cur = cn_label(labels, jT * Ni + iT);
            if (cur > (unsigned)R) cur = 0;
        }
        // this lane's event (one of start, end, transition) and its occupancy key; -1: none
        int ev = -1, occ = -1, arr = -1;
        unsigned tau = 0;
        int2 ns = s;
        if (status == 0u) {
            if (valid) {
                ev = (int)cur;
                if (t) occ = o_count + (int)(cur * R1 + cur);
                ns.x = cur ? (int)(1u << (cur - 1)) : 0;
                ns.y = (int)((unsigned)t | cur << 16 | cur << 21 | 1u << 26);
            }
        } else if (status == 1u) {
            if (!valid) {
                ev = o_end + (int)src;
                ns.y = (int)(w & ~(3u << 26) | 2u << 26);
            } else {
                ev = o_trans + (int)(prev * R1 + cur);
                occ = o_count + (int)(src * R1 + cur);
                if (cur && !((unsigned)s.x >> (cur - 1) & 1u)) {
                    tau = (unsigned)t - start;
                    arr = (int)(src * R + cur - 1);
                    ns.x = (int)((unsigned)s.x | 1u << (cur - 1));
                }
                ns.y = (int)(w & ~(31u << 21) | cur << 21);
            }
        }
        unsigned peers = cn_peers(ev);
        if (ev >= 0 && lane == (unsigned)__ffs(peers) - 1) atomicAdd(s32 + ev, (unsigned)__popc(peers));
        peers = cn_peers(occ);
        if (occ >= 0 && lane == (unsigned)__ffs(peers) - 1) atomicAdd(s32 + occ, (unsigned)__popc(peers));
        if (__any_sync(CN_FULL, arr >= 0)) {
            const int hk = arr >= 0 ? arr * NB + bin_right(tau_edges, ntau, (double)tau) : -1;
            peers = cn_peers(hk);
            if (hk >= 0) {
                const unsigned long long tt = tau;
                atomicAdd(s_sum + arr, tt);
                atomicAdd(s_sum + R1 * R + arr, tt * tt);
                if (lane == (unsigned)__ffs(peers) - 1) {
                    const unsigned n = (unsigned)__popc(peers);
                    atomicAdd(g_hist + hk, (unsigned long long)n);
                    atomicAdd(s32 + o_arr + arr, n);
                }
            }
        }
        if (in && (ns.x != s.x || ns.y != s.y || t == 0)) __stcs(state + p, ns);
    }
    __syncthreads();
    for (int k = threadIdx.x; k < n32; k += CN_BLOCK)
        if (s32[k]) atomicAdd(stats + k, (unsigned long long)s32[k]);
    for (int k = threadIdx.x; k < n64; k += CN_BLOCK)
        if (s_sum[k]) atomicAdd(stats + n32 + k, s_sum[k]);
}

cudaError_t launch_connect(long long nP, int Nj, int Ni, const uint8_t* labels, int R, const int2* cell,
                           const int8_t* mask, int t, int32_t* state, int ntau, const double* tau_edges,
                           int64_t* stats, cudaStream_t st)
{
    // one wave of resident blocks, grid-strided (the statistics are integers: the grid does not change them)
    const size_t smem = connect_smem(R);
    cudaError_t e;
    int dev = 0, nsm = 0, per_sm = 0;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess ||
        (e = cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess ||
        (e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_connect, CN_BLOCK, smem)) != cudaSuccess)
        return e;
    const long long tiles = (nP + CN_BLOCK - 1) / CN_BLOCK, wave = (long long)nsm * (per_sm < 1 ? 1 : per_sm);
    const int grid = (int)(tiles < wave ? tiles : wave);
    k_connect<<<grid, CN_BLOCK, smem, st>>>(nP, Nj, Ni, labels, R, cell, mask, t, reinterpret_cast<int2*>(state), ntau,
                                            tau_edges, reinterpret_cast<unsigned long long*>(stats));
    return cudaGetLastError();
}

}  // namespace st
