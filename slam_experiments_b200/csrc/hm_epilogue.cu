// Epilogues over packed top-2 keys: shard/split merge, Lowe ratio test, mutual
// cross-check, the reference's distance filter, ordered stream compaction.
//
//  - merge: top-k of a union = top-k of the per-set top-k's (SURVEY.md 8e);
//    unsigned min over (dist << 32 | idx) is cv2's tie order.
//  - ratio: integer LUT form of `m.distance < ratio * n.distance` (float64 on the
//    host, see oracle/hamming_oracle.py:ratio_lut) so bit-exactness never depends
//    on GPU floating point.
//  - mutual: cv2.BFMatcher(crossCheck=True).match == strict mutual NN with
//    lowest-index ties both ways (SURVEY.md E4); the reverse pass is a k-NN with
//    roles swapped.
//  - distance filter: /root/reference/feature_matchers.py:41-43,
//    keep d < max(2 * min_d, dist_threshold) (strict).
#include <string.h>

#include "hm_common.cuh"

namespace hm {

namespace {

__global__ void __launch_bounds__(256) hm_merge_top2_kernel(const unsigned long long* __restrict__ keys,
                                                            int groups, long long rows,
                                                            unsigned long long* __restrict__ out)
{
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows) return;
    unsigned long long k1 = kNoMatch, k2 = kNoMatch;
    fold_partials(keys, groups, rows * 2, r, k1, k2);
    *reinterpret_cast<ulonglong2*>(out + r * 2) = make_ulonglong2(k1, k2);
}

// ---- cross-GPU exchange + merge as a stand-alone launch (hm_exchange_merge) ---------------------------
struct ExchangeParams {
    const unsigned long long* local;   // [local_groups][rows][2]
    int local_groups;
    unsigned long long* out;
    long long rows;
    ExchangeArgs x;
};

__global__ void __launch_bounds__(kExchangeRows) hm_exchange_merge_kernel(const ExchangeParams P)
{
    const long long r = (long long)blockIdx.x * kExchangeRows + threadIdx.x;
    const bool has_row = r < P.rows;
    ulonglong2 mine = make_ulonglong2(kNoMatch, kNoMatch);
    if (has_row) fold_partials(P.local, P.local_groups, P.rows * 2, r, mine.x, mine.y);   // fold the train splits
    const ulonglong2 k = exchange_and_merge(P.x, r, has_row, mine, blockIdx.x);
    if (has_row) *reinterpret_cast<ulonglong2*>(P.out + r * 2) = k;
}

constexpr int kFilterThreads = 1024;

struct FilterParams {
    const unsigned long long* fwd;
    const unsigned long long* bwd;
    long long nq, nt;
    unsigned flags;
    int thr_ceil;                    // ceil(dist_threshold), exact integer form of the float compare
    int* out_q;
    int* out_t;
    int* out_d;
    int* out_count;
    const int* slot_of;              // [batch][nt] candidate slots + 1 (SelectArgs), null = bwd indexed by train row
    const unsigned char* mutual;     // [batch][nq] per-query mutual flags (keyframe database), null = use bwd
    RatioLut lut;
};

// Ordered block scan of one flag per thread (all kFilterThreads threads call it): returns how many threads below this
// one have `keep` set and, through `total`, how many in the CTA do.  warp_sums is shared scratch of 32 ints; the caller
// synchronises before warp_sums is written again.
__device__ __forceinline__ int ordered_scan(int keep, int* warp_sums, int& total)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const unsigned ballot = __ballot_sync(0xFFFFFFFFu, keep);
    const int prefix = __popc(ballot & ((1u << lane) - 1));
    if (lane == 0) warp_sums[wid] = __popc(ballot);
    __syncthreads();
    int v = lane < (kFilterThreads / 32) ? warp_sums[lane] : 0;
    int incl = v;
    for (int o = 1; o < 32; o <<= 1) {
        int n = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= o) incl += n;
    }
    total = __shfl_sync(0xFFFFFFFFu, incl, 31);
    return __shfl_sync(0xFFFFFFFFu, incl - v, wid) + prefix;
}

// One CTA per problem: rows are visited in order so the output stays sorted by queryIdx.
__global__ void __launch_bounds__(kFilterThreads) hm_filter_kernel(const FilterParams P)
{
    __shared__ int warp_sums[32];
    __shared__ int s_base;
    __shared__ unsigned s_min;
    const int tid = threadIdx.x, lane = tid & 31;
    const int b = blockIdx.x;
    const unsigned long long* fwd = P.fwd + (long long)b * P.nq * 2;
    const unsigned long long* bwd = P.bwd ? P.bwd + (long long)b * P.nt * 2 : nullptr;
    int* oq = P.out_q + (long long)b * P.nq;
    int* ot = P.out_t + (long long)b * P.nq;
    int* od = P.out_d + (long long)b * P.nq;

    int limit = 0x7FFFFFFF;
    if (P.flags & HM_FLAG_DIST_THRESHOLD) {
        if (tid == 0) s_min = 0xFFFFFFFFu;
        __syncthreads();
        unsigned m = 0xFFFFFFFFu;
        for (long long r = tid; r < P.nq; r += kFilterThreads) {
            const unsigned long long k1 = fwd[r * 2];
            if (k1 != kNoMatch) m = min(m, (unsigned)(k1 >> 32));
        }
        for (int o = 16; o; o >>= 1) m = min(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
        if (lane == 0) atomicMin(&s_min, m);
        __syncthreads();
        const unsigned mn = s_min;
        limit = mn == 0xFFFFFFFFu ? 0 : max((int)(2 * mn), P.thr_ceil);
    }
    if (tid == 0) s_base = 0;
    __syncthreads();

    for (long long r0 = 0; r0 < P.nq; r0 += kFilterThreads) {
        const long long r = r0 + tid;
        int keep = 0, t1 = 0, d1 = 0;
        if (r < P.nq) {
            const ulonglong2 k = *reinterpret_cast<const ulonglong2*>(fwd + r * 2);
            keep = k.x != kNoMatch;
            t1 = (int)(unsigned)(k.x & 0xFFFFFFFFull);
            d1 = (int)(k.x >> 32);
            if (keep && (P.flags & HM_FLAG_RATIO)) {
                keep = (k.y != kNoMatch) && d1 < (int)P.lut.v[min((unsigned)(k.y >> 32), 256u)];
            }
            if (keep && (P.flags & HM_FLAG_MUTUAL) && P.mutual) {
                keep = P.mutual[(long long)b * P.nq + r] != 0;
            } else if (keep && (P.flags & HM_FLAG_MUTUAL)) {
                // bwd is indexed by train row, or -- after the candidate pass -- by the row's candidate slot (a row
                // that reaches this line passed the ratio test, so the k-NN kernel gave its best train row a slot)
                const long long slot = P.slot_of ? (long long)P.slot_of[(long long)b * P.nt + t1] - 1 : (long long)t1;
                keep = slot >= 0 && (long long)(bwd[slot * 2] & 0xFFFFFFFFull) == r;
            }
            if (keep && (P.flags & HM_FLAG_DIST_THRESHOLD)) keep = d1 < limit;
        }
        int total;
        const int offset = ordered_scan(keep, warp_sums, total);
        const int base = s_base;
        if (keep) {
            const int pos = base + offset;
            oq[pos] = (int)r;
            ot[pos] = t1;
            od[pos] = d1;
        }
        __syncthreads();
        if (tid == 0) s_base = base + total;
        __syncthreads();
    }
    if (tid == 0) P.out_count[b] = s_base;
}

// ---- keyframe database: mutual check of one shard (hm_db_mutual_flags) -------------------------------------------
// The mutual check asks, for the best database row t1 of every query, which query of the batch is nearest to t1.  The
// shard that holds t1 answers: select lists its queries in query order (one CTA, the filter's ordered scan), a top-1
// k-NN of the listed shard rows against the query batch follows (hm_api.cu), and resolve marks each listed query that
// is its row's nearest query.  A row named by several queries is listed once per query: an extra row of an nq-row pass
// costs less than a table indexed by database row.
struct DbSelectParams {
    const unsigned long long* keys;  // [nq][2] global top-2
    long long nq;
    unsigned long long row_lo, row_hi;
    int use_ratio;
    const uint8_t* shard_bits;
    long long t_stride;
    int* list;                       // [nq] local shard rows
    int* owner;                      // [nq] the query that named each row
    int* count;
    uint8_t* gathered;               // [nq][32] or null (the kind::mxf4 k-NN kernel gathers through `list` itself)
    unsigned char* flags;            // [nq]
    RatioLut lut;
};

__global__ void __launch_bounds__(kFilterThreads) hm_db_select_kernel(const DbSelectParams P)
{
    __shared__ int warp_sums[32];
    __shared__ int s_base;
    const int tid = threadIdx.x;
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (long long r0 = 0; r0 < P.nq; r0 += kFilterThreads) {
        const long long r = r0 + tid;
        int own = 0;
        unsigned long long t1 = 0;
        if (r < P.nq) {
            const ulonglong2 k = *reinterpret_cast<const ulonglong2*>(P.keys + r * 2);
            t1 = k.x & 0xFFFFFFFFull;
            own = k.x != kNoMatch && t1 >= P.row_lo && t1 < P.row_hi;
            if (own && P.use_ratio)     // the filter's ratio test: a row it drops needs no backward answer
                own = k.y != kNoMatch && (unsigned)(k.x >> 32) < (unsigned)P.lut.v[min((unsigned)(k.y >> 32), 256u)];
            P.flags[r] = 0;
        }
        int total;
        const int offset = ordered_scan(own, warp_sums, total);
        const int base = s_base;
        if (own) {
            const int s = base + offset;
            const long long local = (long long)(t1 - P.row_lo);
            P.list[s] = (int)local;
            P.owner[s] = (int)r;
            if (P.gathered) {
                const uint4* src = reinterpret_cast<const uint4*>(P.shard_bits + local * P.t_stride);
                uint4* dst = reinterpret_cast<uint4*>(P.gathered + (long long)s * HM_DESC_BYTES);
                dst[0] = src[0];
                dst[1] = src[1];
            }
        }
        __syncthreads();
        if (tid == 0) s_base = base + total;
        __syncthreads();
    }
    const int n = s_base;
    if (tid == 0) *P.count = n;
    if (P.gathered) {                // the dense k-NN pass reads all nq rows: keep the unused ones defined
        for (long long s = n + tid; s < P.nq; s += kFilterThreads) {
            uint4* dst = reinterpret_cast<uint4*>(P.gathered + s * HM_DESC_BYTES);
            dst[0] = make_uint4(0, 0, 0, 0);
            dst[1] = make_uint4(0, 0, 0, 0);
        }
    }
}

__global__ void __launch_bounds__(256) hm_db_resolve_kernel(const int* __restrict__ owner, const int* __restrict__ count,
                                                            const unsigned long long* __restrict__ best,
                                                            unsigned char* __restrict__ flags)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= *count) return;
    const int q = owner[s];
    const unsigned long long k = best[(long long)s * 2];
    if (k != kNoMatch && (long long)(k & 0xFFFFFFFFull) == q) flags[q] = 1;
}

}  // namespace

int launch_merge_top2(const unsigned long long* keys, int groups, long long rows, unsigned long long* out,
                      cudaStream_t stream)
{
    if (rows <= 0) return HM_OK;
    const int threads = 64;      // few rows: spread them over many SMs
    const long long blocks = ceil_div(rows, threads);
    hm_merge_top2_kernel<<<(unsigned)blocks, threads, 0, stream>>>(keys, groups, rows, out);
    HM_CUDA_CHECK(cudaGetLastError());
    return HM_OK;
}

size_t exchange_bytes(long long max_rows, int world)
{
    return exchange_keys_bytes(max_rows, world) + (size_t)world * exchange_blocks(max_rows) * sizeof(unsigned) + 256;
}

int fill_exchange_args(ExchangeArgs* x, int world, int rank, void* const* peers, long long max_rows, unsigned epoch,
                       long long rows)
{
    if (world < 1 || world > kMaxWorld || rank < 0 || rank >= world || rows > max_rows || rows <= 0 || epoch == 0 || !peers) {
        set_error("exchange: bad arguments (world %d rank %d rows %lld max_rows %lld epoch %u)", world, rank, rows,
                  max_rows, epoch);
        return HM_ERR_INVALID_ARGUMENT;
    }
    memset(x, 0, sizeof(*x));
    x->world = world; x->rank = rank; x->epoch = epoch; x->max_rows = max_rows;
    for (int i = 0; i < world; ++i) {
        if (!peers[i]) {
            set_error("exchange: null peer buffer %d", i);
            return HM_ERR_INVALID_ARGUMENT;
        }
        x->peer[i] = static_cast<unsigned char*>(peers[i]);
    }
    return HM_OK;
}

int launch_exchange_merge(const unsigned long long* local_keys, int local_groups, long long rows, int world, int rank,
                          void* const* peers, long long max_rows, unsigned epoch, unsigned long long* out,
                          cudaStream_t stream)
{
    ExchangeParams P{};
    if (local_groups < 1) {
        set_error("hm_exchange_merge: local_groups < 1");
        return HM_ERR_INVALID_ARGUMENT;
    }
    int rc = fill_exchange_args(&P.x, world, rank, peers, max_rows, epoch, rows);
    if (rc != HM_OK) return rc;
    P.local = local_keys; P.local_groups = local_groups; P.out = out; P.rows = rows;
    // One CTA and one flag per 256-row block that holds rows.  `rows` is the replicated query's size, identical on
    // every rank, and the k-NN kernel's fused exchange uses the same blocks: ranks may mix the two kernels (a rank
    // without a prepared shard runs this one) and still post / wait on exactly the same flags.
    hm_exchange_merge_kernel<<<(unsigned)ceil_div(rows, kExchangeRows), kExchangeRows, 0, stream>>>(P);
    HM_CUDA_CHECK(cudaGetLastError());
    return HM_OK;
}

int launch_filter(const unsigned long long* fwd, long long nq, const unsigned long long* bwd, long long nt,
                  int batch, unsigned flags, const RatioLut& lut, int thr_ceil, int* out_q, int* out_t,
                  int* out_d, int* out_count, cudaStream_t stream, const int* slot_of,
                  const unsigned char* mutual_flags)
{
    if (batch <= 0) return HM_OK;
    FilterParams P{};
    P.slot_of = slot_of;
    P.mutual = mutual_flags;
    P.fwd = fwd; P.bwd = bwd; P.nq = nq; P.nt = nt; P.flags = flags;
    P.out_q = out_q; P.out_t = out_t; P.out_d = out_d; P.out_count = out_count;
    P.lut = lut;
    P.thr_ceil = thr_ceil;
    hm_filter_kernel<<<batch, kFilterThreads, 0, stream>>>(P);
    HM_CUDA_CHECK(cudaGetLastError());
    return HM_OK;
}

int launch_db_select(const unsigned long long* keys, long long nq, unsigned long long row_lo, unsigned long long row_hi,
                     int use_ratio, const RatioLut& lut, const uint8_t* shard_bits, long long t_stride, int* list,
                     int* owner, int* count, uint8_t* gathered, unsigned char* flags, cudaStream_t stream)
{
    if (nq <= 0) return HM_OK;
    DbSelectParams P{};
    P.keys = keys; P.nq = nq; P.row_lo = row_lo; P.row_hi = row_hi; P.use_ratio = use_ratio;
    P.shard_bits = shard_bits; P.t_stride = t_stride;
    P.list = list; P.owner = owner; P.count = count; P.gathered = gathered; P.flags = flags;
    P.lut = lut;
    hm_db_select_kernel<<<1, kFilterThreads, 0, stream>>>(P);
    HM_CUDA_CHECK(cudaGetLastError());
    return HM_OK;
}

int launch_db_resolve(const int* owner, const int* count, const unsigned long long* best, long long nq,
                      unsigned char* flags, cudaStream_t stream)
{
    if (nq <= 0) return HM_OK;
    hm_db_resolve_kernel<<<(unsigned)ceil_div(nq, 256), 256, 0, stream>>>(owner, count, best, flags);
    HM_CUDA_CHECK(cudaGetLastError());
    return HM_OK;
}

// ---- consumer of the match list (SURVEY.md 8f rank 2) ------------------------------------------------
// /root/reference/utils.py:13-19 and :41-47 build two point lists with a Python loop over the matches
// (source_frame.features[m.trainIdx].position, query_frame.features[m.queryIdx].position); here the
// keypoint positions stay resident next to the descriptors and the two packed (M, 2) arrays are gathered
// on the device from the match list the filter kernel produced.
struct GatherParams {
    const int* q_idx;
    const int* t_idx;
    const int* count;
    long long stride;                // match-list elements per problem
    const int2* query_pts;           // [batch][nq]
    const int2* train_pts;           // [batch][nt]
    long long nq, nt;
    int2* out_query;
    int2* out_train;
};

__global__ void __launch_bounds__(256) hm_gather_points_kernel(const GatherParams P)
{
    const int b = blockIdx.y;
    const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= P.count[b]) return;
    const long long o = (long long)b * P.stride + m;
    const int q = P.q_idx[o], t = P.t_idx[o];
    P.out_query[o] = P.query_pts[(long long)b * P.nq + q];
    P.out_train[o] = P.train_pts[(long long)b * P.nt + t];
}

int launch_gather_points(const int* q_idx, const int* t_idx, const int* count, long long stride, int batch,
                         const int* query_pts, long long nq, const int* train_pts, long long nt, int* out_query,
                         int* out_train, cudaStream_t stream)
{
    if (batch <= 0 || stride <= 0) return HM_OK;
    GatherParams P{};
    P.q_idx = q_idx; P.t_idx = t_idx; P.count = count; P.stride = stride;
    P.query_pts = reinterpret_cast<const int2*>(query_pts);
    P.train_pts = reinterpret_cast<const int2*>(train_pts);
    P.nq = nq; P.nt = nt;
    P.out_query = reinterpret_cast<int2*>(out_query);
    P.out_train = reinterpret_cast<int2*>(out_train);
    dim3 grid((unsigned)ceil_div(stride, 256), (unsigned)batch);
    hm_gather_points_kernel<<<grid, 256, 0, stream>>>(P);
    HM_CUDA_CHECK(cudaGetLastError());
    return HM_OK;
}

// ---- detection mask (SURVEY.md 8f rank 4) --------------------------------------------------------------
// /root/reference/utils.py:58-74: mask = full(shape, inner ? 0 : 255); for every feature
// cv2.rectangle(mask, pt - r, pt + r, inner ? 255 : 0, FILLED) -- inclusive corners, clipped to the image.
// All rectangles write the same value, so the result does not depend on the order: one warp per feature,
// after one fill.  HBM-bound on the fill (h * w bytes); the rectangles touch n * (2r+1)^2 bytes.
struct MaskParams {
    const int2* pts;
    long long n;
    int radius, h, w;
    long long row_stride;
    unsigned char* mask;
    unsigned char value;
};

__global__ void __launch_bounds__(256) hm_mask_fill_kernel(unsigned char* mask, int h, int w, long long row_stride, unsigned char v)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)h * w) return;
    mask[(i / w) * row_stride + (i % w)] = v;
}

__global__ void __launch_bounds__(256) hm_mask_rect_kernel(const MaskParams P)
{
    const long long f = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (f >= P.n) return;
    const int lane = threadIdx.x & 31;
    const int2 p = P.pts[f];
    // 64-bit corners: positions near INT_MAX must clip, not wrap
    const long long x0 = max((long long)p.x - P.radius, 0ll), x1 = min((long long)p.x + P.radius, (long long)P.w - 1);
    const long long y0 = max((long long)p.y - P.radius, 0ll), y1 = min((long long)p.y + P.radius, (long long)P.h - 1);
    if (x0 > x1 || y0 > y1) return;
    const long long wd = x1 - x0 + 1, cells = wd * (y1 - y0 + 1);
    for (long long c = lane; c < cells; c += 32) P.mask[(y0 + c / wd) * P.row_stride + x0 + c % wd] = P.value;
}

int launch_rasterize_mask(const int* pts, long long n, int radius, int inner, unsigned char* mask, int h, int w,
                          long long row_stride, cudaStream_t stream)
{
    if (h <= 0 || w <= 0) return HM_OK;
    const long long cells = (long long)h * w;
    hm_mask_fill_kernel<<<(unsigned)ceil_div(cells, 256), 256, 0, stream>>>(mask, h, w, row_stride, inner ? 0 : 255);
    HM_CUDA_CHECK(cudaGetLastError());
    if (n > 0) {
        MaskParams P{};
        P.pts = reinterpret_cast<const int2*>(pts); P.n = n; P.radius = radius; P.h = h; P.w = w;
        P.row_stride = row_stride; P.mask = mask; P.value = inner ? 255 : 0;
        hm_mask_rect_kernel<<<(unsigned)ceil_div(n, 8), 256, 0, stream>>>(P);
        HM_CUDA_CHECK(cudaGetLastError());
    }
    return HM_OK;
}

}  // namespace hm
