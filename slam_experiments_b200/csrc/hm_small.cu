// Small problems in ONE launch: the whole match() pipeline of /root/reference/feature_matchers.py:32-44 (and the
// ratio / mutual extensions of SURVEY.md 8a row P) for frames of up to 1024 descriptors each -- the reference's own
// configuration is 200 (slam.py:23).
//
// At this size the work is ~6 us of GPU time behind five launches, two copies and a stream synchronisation
// (hm_match_fused + the CUDA graph of hm_match_host: 39-44 us per 200 x 200 call).  Here ONE thread-block cluster of
// 8 CTAs does everything and the host never calls into the driver after the launch:
//   - each CTA reads 1/8 of both descriptor sets straight from the caller's pinned, device-mapped staging buffer
//     (12.8 KB over PCIe in total, every byte once) into its shared memory; after a cluster barrier every CTA copies
//     the other seven slices through distributed shared memory, so all 8 SMs hold both sets;
//   - forward k-NN, XOR + POPC (the POPC pipe issues 16 per clock per SM, hence 8 SMs): one WARP per query row, lanes
//     stride over the train rows with a packed (distance << 32 | trainIdx) top-2 each, merged by a warp-shuffle
//     top-2 reduction (unsigned min = cv2's order);
//   - with HM_FLAG_MUTUAL the same pass with the roles swapped (top-1), from the same shared-memory copies;
//   - CTA 0 collects the keys over DSMEM and runs the ratio LUT / mutual / distance-threshold filter with the ordered
//     compaction (block scan over the query rows);
//   - the match list is written to mapped host memory, followed by a system-scope release store of the call's epoch;
//     the host polls that word (bounded, with cudaStreamQuery as the failure check) instead of synchronising.
#include <cooperative_groups.h>

#include <mutex>

#include "hm_common.cuh"

namespace cg = cooperative_groups;

namespace hm {
namespace {

constexpr int kSmallThreads = 512;
constexpr int kSmallWarps = kSmallThreads / 32;
constexpr int kSmallCluster = 8;

struct SmallParams {
    const uint4* q;                  // [nq][2] uint4 (32-byte rows, contiguous)
    const uint4* t;                  // [nt][2]
    int nq, nt;
    unsigned flags;
    int thr_ceil;
    int* out;                        // mapped host memory: [count, epoch, pad, pad][q nq][t nq][d nq]
    unsigned epoch;
    RatioLut lut;
};

__device__ __forceinline__ unsigned dist_row(const uint4 a0, const uint4 a1, const uint4 b0, const uint4 b1)
{
    return __popc(a0.x ^ b0.x) + __popc(a0.y ^ b0.y) + __popc(a0.z ^ b0.z) + __popc(a0.w ^ b0.w) +
           __popc(a1.x ^ b1.x) + __popc(a1.y ^ b1.y) + __popc(a1.z ^ b1.z) + __popc(a1.w ^ b1.w);
}

// warp-wide top-2 of per-lane (k1 <= k2) pairs: butterfly over 5 shuffle rounds, every lane ends with the result
__device__ __forceinline__ void warp_top2(unsigned long long& k1, unsigned long long& k2)
{
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        const unsigned long long a = __shfl_xor_sync(0xFFFFFFFFu, k1, o), b = __shfl_xor_sync(0xFFFFFFFFu, k2, o);
        top2_insert(k1, k2, a);
        top2_insert(k1, k2, b);
    }
}

// rows [lo, hi) of `n` that cluster rank `rank` owns
__device__ __forceinline__ void slice(int n, int rank, int& lo, int& hi)
{
    const int per = (n + kSmallCluster - 1) / kSmallCluster;
    lo = min(rank * per, n);
    hi = min(lo + per, n);
}

__global__ void __cluster_dims__(kSmallCluster, 1, 1) __launch_bounds__(kSmallThreads, 1) hm_small_match_kernel(const SmallParams P)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint4* sq = reinterpret_cast<uint4*>(smem_raw);                       // [nq][2]
    uint4* st = sq + 2 * P.nq;                                            // [nt][2]
    ulonglong2* fwd = reinterpret_cast<ulonglong2*>(st + 2 * P.nt);       // [nq] top-2 keys
    unsigned long long* bwd = reinterpret_cast<unsigned long long*>(fwd + P.nq);   // [nt] best query key
    __shared__ int warp_sums[32];
    __shared__ int s_base;
    __shared__ unsigned s_min;

    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int q_lo, q_hi, t_lo, t_hi;
    slice(P.nq, rank, q_lo, q_hi);
    slice(P.nt, rank, t_lo, t_hi);
    // 1. this CTA's slices from (mapped host) memory
    for (int i = 2 * q_lo + tid; i < 2 * q_hi; i += kSmallThreads) sq[i] = P.q[i];
    for (int i = 2 * t_lo + tid; i < 2 * t_hi; i += kSmallThreads) st[i] = P.t[i];
    if (tid == 0) { s_base = 0; s_min = 0xFFFFFFFFu; }
    cluster.sync();
    // 2. the other CTAs' slices over distributed shared memory
    for (int r = 1; r < kSmallCluster; ++r) {
        const int peer = (rank + r) % kSmallCluster;
        int lo, hi;
        slice(P.nq, peer, lo, hi);
        const uint4* pq = cluster.map_shared_rank(sq, peer);
        for (int i = 2 * lo + tid; i < 2 * hi; i += kSmallThreads) sq[i] = pq[i];
        slice(P.nt, peer, lo, hi);
        const uint4* pt = cluster.map_shared_rank(st, peer);
        for (int i = 2 * lo + tid; i < 2 * hi; i += kSmallThreads) st[i] = pt[i];
    }
    __syncthreads();

    // 3. forward: nearest two train rows of this CTA's query rows
    for (int r = q_lo + warp; r < q_hi; r += kSmallWarps) {
        const uint4 a0 = sq[2 * r], a1 = sq[2 * r + 1];
        unsigned long long k1 = kNoMatch, k2 = kNoMatch;
        for (int c = lane; c < P.nt; c += 32)
            top2_insert(k1, k2, ((unsigned long long)dist_row(a0, a1, st[2 * c], st[2 * c + 1]) << 32) | (unsigned)c);
        warp_top2(k1, k2);
        if (lane == 0) fwd[r] = make_ulonglong2(k1, k2);
    }
    //    swapped pass of the mutual check: nearest query row of this CTA's train rows
    if (P.flags & HM_FLAG_MUTUAL) {
        for (int c = t_lo + warp; c < t_hi; c += kSmallWarps) {
            const uint4 b0 = st[2 * c], b1 = st[2 * c + 1];
            unsigned long long k = kNoMatch;
            for (int r = lane; r < P.nq; r += 32) {
                const unsigned long long key = ((unsigned long long)dist_row(sq[2 * r], sq[2 * r + 1], b0, b1) << 32) | (unsigned)r;
                k = key < k ? key : k;
            }
#pragma unroll
            for (int o = 16; o; o >>= 1) {
                const unsigned long long other = __shfl_xor_sync(0xFFFFFFFFu, k, o);
                k = other < k ? other : k;
            }
            if (lane == 0) bwd[c] = k;
        }
    }
    cluster.sync();          // every CTA's keys are in its shared memory
    if (rank != 0) {
        cluster.sync();      // stay resident until CTA 0 has read them
        return;
    }
    // 4. CTA 0: collect the keys
    for (int r = 1; r < kSmallCluster; ++r) {
        int lo, hi;
        slice(P.nq, r, lo, hi);
        const ulonglong2* pf = cluster.map_shared_rank(fwd, r);
        for (int i = lo + tid; i < hi; i += kSmallThreads) fwd[i] = pf[i];
        if (P.flags & HM_FLAG_MUTUAL) {
            slice(P.nt, r, lo, hi);
            const unsigned long long* pb = cluster.map_shared_rank(bwd, r);
            for (int i = lo + tid; i < hi; i += kSmallThreads) bwd[i] = pb[i];
        }
    }
    cluster.sync();          // peers may exit
    __syncthreads();

    // the reference's distance filter needs the smallest best distance first (feature_matchers.py:41-43)
    int limit = 0x7FFFFFFF;
    if (P.flags & HM_FLAG_DIST_THRESHOLD) {
        unsigned m = 0xFFFFFFFFu;
        for (int r = tid; r < P.nq; r += kSmallThreads)
            if (fwd[r].x != kNoMatch) m = min(m, (unsigned)(fwd[r].x >> 32));
        m = __reduce_min_sync(0xFFFFFFFFu, m);
        if (lane == 0) atomicMin(&s_min, m);
        __syncthreads();
        const unsigned mn = s_min;
        limit = mn == 0xFFFFFFFFu ? 0 : max((int)(2 * mn), P.thr_ceil);
    }

    int* oq = P.out + 4;
    int* ot = oq + P.nq;
    int* od = ot + P.nq;
    for (int r0 = 0; r0 < P.nq; r0 += kSmallThreads) {      // ordered compaction, as hm_filter_kernel
        const int r = r0 + tid;
        int keep = 0, t1 = 0, d1 = 0;
        if (r < P.nq) {
            const ulonglong2 k = fwd[r];
            keep = k.x != kNoMatch;
            t1 = (int)(unsigned)(k.x & 0xFFFFFFFFull);
            d1 = (int)(k.x >> 32);
            if (keep && (P.flags & HM_FLAG_RATIO)) keep = (k.y != kNoMatch) && d1 < (int)P.lut.v[min((unsigned)(k.y >> 32), 256u)];
            if (keep && (P.flags & HM_FLAG_MUTUAL)) keep = (int)(bwd[t1] & 0xFFFFFFFFull) == r;
            if (keep && (P.flags & HM_FLAG_DIST_THRESHOLD)) keep = d1 < limit;
        }
        const unsigned ballot = __ballot_sync(0xFFFFFFFFu, keep);
        const int prefix = __popc(ballot & ((1u << lane) - 1));
        if (lane == 0) warp_sums[warp] = __popc(ballot);
        __syncthreads();
        const int v = lane < kSmallWarps ? warp_sums[lane] : 0;
        int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int n = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= o) incl += n;
        }
        const int wbase = __shfl_sync(0xFFFFFFFFu, incl - v, warp);
        const int total = __shfl_sync(0xFFFFFFFFu, incl, 31);
        const int base = s_base;
        if (keep) {
            const int pos = base + wbase + prefix;
            oq[pos] = r;
            ot[pos] = t1;
            od[pos] = d1;
        }
        __syncthreads();
        if (tid == 0) s_base = base + total;
        __syncthreads();
    }
    // publish: every thread's result stores are ordered before the epoch word by the fence + barrier
    __threadfence_system();
    __syncthreads();
    if (tid == 0) {
        P.out[0] = s_base;
        asm volatile("st.release.sys.global.u32 [%0], %1;\n" ::"l"(P.out + 1), "r"(P.epoch) : "memory");
    }
}

}  // namespace

size_t small_smem_bytes(long long nq, long long nt) { return (size_t)(nq + nt) * 32 + (size_t)nq * 16 + (size_t)nt * 8; }

bool small_match_eligible(long long nq, long long nt)
{
    return nq > 0 && nt > 0 && nq <= HM_SMALL_MAX_ROWS && nt <= HM_SMALL_MAX_ROWS && nq * nt <= HM_SMALL_MAX_PAIRS;
}

// q / t: device-accessible pointers (device memory or mapped pinned host memory), 32-byte rows, 16-byte aligned;
// out_mapped: mapped pinned host memory, 16 + 12 nq bytes
int launch_small_match(const uint8_t* q, long long nq, const uint8_t* t, long long nt, unsigned flags, const RatioLut& lut,
                       int thr_ceil, int* out_mapped, unsigned epoch, cudaStream_t stream)
{
    static std::mutex mu;                     // the > 48 KB opt-in is per device; one process may drive several
    static bool attr_done[64] = {};
    int dev = 0;
    HM_CUDA_CHECK(cudaGetDevice(&dev));
    {
        std::lock_guard<std::mutex> lock(mu);
        if (dev < 0 || dev >= 64 || !attr_done[dev]) {
            HM_CUDA_CHECK(cudaFuncSetAttribute(hm_small_match_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               (int)small_smem_bytes(HM_SMALL_MAX_ROWS, HM_SMALL_MAX_ROWS)));
            if (dev >= 0 && dev < 64) attr_done[dev] = true;
        }
    }
    SmallParams P{};
    P.q = reinterpret_cast<const uint4*>(q); P.t = reinterpret_cast<const uint4*>(t);
    P.nq = (int)nq; P.nt = (int)nt; P.flags = flags; P.thr_ceil = thr_ceil; P.out = out_mapped; P.epoch = epoch; P.lut = lut;
    hm_small_match_kernel<<<kSmallCluster, kSmallThreads, small_smem_bytes(nq, nt), stream>>>(P);
    HM_CUDA_CHECK(cudaGetLastError());
    return HM_OK;
}

}  // namespace hm
