// Shared device/host helpers for the Hamming matcher kernels (sm_100a).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "hm_matcher.h"

namespace hm {

constexpr unsigned long long kNoMatch = 0xFFFFFFFFFFFFFFFFull;

// thread-local error string behind hm_last_error()
void set_error(const char* fmt, ...);

#define HM_CUDA_CHECK(expr)                                                              \
    do {                                                                                 \
        cudaError_t _e = (expr);                                                         \
        if (_e != cudaSuccess) {                                                         \
            hm::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),        \
                          __FILE__, __LINE__);                                           \
            return HM_ERR_CUDA;                                                          \
        }                                                                                \
    } while (0)

// One k-NN problem family: `batch` problems of identical shape.
struct KnnProblem {
    const uint8_t* q;
    const uint8_t* t;
    long long nq, nt;
    long long q_stride, t_stride;             // bytes between rows
    long long q_batch_stride, t_batch_stride; // bytes between problems
    int batch;
    unsigned long long train_base;            // added to every trainIdx
    bool top1;                                // only the nearest neighbour is needed (second key may be HM_NO_MATCH)
    const struct SelectArgs* select;          // tensor-core kind::mxf4 launches only: see SelectArgs
};

// packed query descriptors handed to the tensor-core launcher (kind::mxf4 expands them inside the k-NN kernel)
struct QueryBits {
    const uint8_t* bits;
    long long stride, batch_stride;
    // optional gather + device-side row count (TcParams::q_index / nq_dyn): the candidate pass of the mutual check
    const int* index;
    long long index_batch_stride;
    const int* nq_dyn;
};

struct RatioLut {
    unsigned short v[257];
};

// A selection of train rows as ascending, disjoint, non-empty runs [lo, hi) of rows (hm_knn2_resident_runs,
// hm_knn2_runs).  The device array holds kRunFields int64 per run: lo, hi, the tiles of 128 rows the runs before it
// touch (their sum of ceil(hi / 128) - floor(lo / 128)) and the rows the runs before it hold.
constexpr int kRunFields = 4;
struct RunArgs {
    const long long* runs;        // device [n_runs][kRunFields]
    int n_runs;
};
// checked on the host from the caller's [n_runs][2] copy: tiles / rows of the whole selection
struct RunTotals {
    long long tiles, rows;
};

// Ratio test + candidate selection on a row's final keys, run by the k-NN kernel that produced them (row P of
// SURVEY.md 8a: /root/reference/feature_matchers.py:34,39 extended by Lowe's test and the mutual check).  A row that
// passes the ratio test marks its best train row as a CANDIDATE column; the swapped pass of the mutual check then
// runs only over the candidate rows (hm_match_fused), not over the whole train set.
struct SelectArgs {
    int* slot_of;        // [batch][nt], zeroed: slot + 1 once the train row is a candidate (-1 while being assigned)
    int* list;           // [batch][nt] candidate train rows, arrival order
    int* count;          // [batch], zeroed
    long long nt;
    int use_ratio;
    RatioLut lut;        // lut[d2] = ceil(ratio * d2): d1 < ratio * d2  <=>  d1 < lut[d2] for integer d1
};

__device__ __forceinline__ void select_candidate(const SelectArgs& S, int b, ulonglong2 k)
{
    if (!S.slot_of || k.x == kNoMatch) return;
    if (S.use_ratio) {
        if (k.y == kNoMatch) return;
        const unsigned d2 = min((unsigned)(k.y >> 32), 256u);
        if (!((unsigned)(k.x >> 32) < (unsigned)S.lut.v[d2])) return;
    }
    const long long t = (long long)(k.x & 0xFFFFFFFFull);
    int* cell = S.slot_of + (long long)b * S.nt + t;
    if (atomicCAS(cell, 0, -1) == 0) {                  // first row that names this train row
        const int s = atomicAdd(S.count + b, 1);
        S.list[(long long)b * S.nt + s] = (int)t;
        atomicExch(cell, s + 1);
    }
}

struct DeviceInfo {
    int device;
    int sm_count;
    int cc_major, cc_minor;
};
// cached per device; returns an hm_status
int device_info(DeviceInfo* out);

// optional event pair recorded around the dominant kernel (hm_profile_events)
void profile_mark(bool start, cudaStream_t stream);

inline __host__ __device__ long long ceil_div(long long a, long long b) { return (a + b - 1) / b; }

// insert `key` into the ascending pair (k1, k2)
__device__ __forceinline__ void top2_insert(unsigned long long& k1, unsigned long long& k2,
                                            unsigned long long key)
{
    unsigned long long hi = key > k1 ? key : k1;
    k1 = key < k1 ? key : k1;
    k2 = hi < k2 ? hi : k2;
}

// ---- in-kernel merge of train splits ("last CTA done" pattern) ---------------------------------------
// Every CTA of a k-NN kernel writes its partial keys to partials[split][row][2]; the CTA that arrives last
// on the per-row-block counter folds all splits and writes the final keys, so no merge kernel is launched.
// min over keys is order independent, so the result does not depend on which CTA is last.
__device__ __forceinline__ bool last_cta_arrives(unsigned* counter, unsigned expected, int* smem_flag)
{
    __threadfence();                       // this thread's partial keys are visible device-wide
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned old = atomicAdd(counter, 1u);
        const int last = old == expected - 1;
        if (last) *counter = 0;            // ready for the next launch on this workspace
        *smem_flag = last;
    }
    __syncthreads();
    const bool last = *smem_flag != 0;
    if (last) __threadfence();
    return last;
}

// top-2 of one row over `groups` partial results (L2-coherent loads, 8 in flight)
__device__ __forceinline__ void fold_partials(const unsigned long long* keys, int groups, long long group_stride,
                                              long long r, unsigned long long& k1, unsigned long long& k2)
{
    int g = 0;
    for (; g + 8 <= groups; g += 8) {
        ulonglong2 k[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) k[j] = __ldcg(reinterpret_cast<const ulonglong2*>(keys + (long long)(g + j) * group_stride + r * 2));
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            top2_insert(k1, k2, k[j].x);
            top2_insert(k1, k2, k[j].y);
        }
    }
    for (; g < groups; ++g) {
        const ulonglong2 k = __ldcg(reinterpret_cast<const ulonglong2*>(keys + (long long)g * group_stride + r * 2));
        top2_insert(k1, k2, k.x);
        top2_insert(k1, k2, k.y);
    }
}

// ---- cross-GPU exchange over symmetric memory (shared by hm_exchange_merge_kernel and the k-NN kernel's
// last-CTA merge).  Symmetric buffer layout, identical on every rank:
//   [2 parities][world slots][max_rows][2] u64 keys | [world][max_rows / 256] u32 epoch flags
constexpr int kMaxWorld = 8;
constexpr int kExchangeRows = 256;          // rows per flag (= rows per CTA of either kernel)

struct ExchangeArgs {
    unsigned char* peer[kMaxWorld];          // peer-mapped base of the symmetric buffer on every rank
    int world, rank;
    unsigned epoch;                          // 1, 2, 3, ... identical on all ranks
    long long max_rows;
};

// row blocks with a flag each; even, because the k-NN kernel launches query blocks in cluster pairs
__host__ __device__ inline long long exchange_blocks(long long max_rows)
{
    return (((max_rows + kExchangeRows - 1) / kExchangeRows) + 1) & ~1ll;
}
__host__ __device__ inline size_t exchange_keys_bytes(long long max_rows, int world)
{
    return (size_t)2 * world * max_rows * 2 * sizeof(unsigned long long);
}

__device__ __forceinline__ void st_release_sys(unsigned* p, unsigned v)
{
    asm volatile("st.release.sys.global.u32 [%0], %1;\n" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned* p)
{
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];\n" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// Called by ALL threads of a CTA that owns row block `block` (rows [block*256, +256)); thread t < 256 passes
// its row's local keys.  Pushes them into slot `rank` of every rank's buffer with peer stores, publishes
// flag[rank][block] = epoch on every rank (release, system scope), waits for every rank's flag for this
// block (acquire; bounded spin -> trap) and returns the merge of all slots for this thread's row.
__device__ __forceinline__ ulonglong2 exchange_and_merge(const ExchangeArgs& X, long long r, bool has_row,
                                                         ulonglong2 mine, long long block)
{
    const int parity = X.epoch & 1;
    const size_t slot_keys = (size_t)X.max_rows * 2;
    const size_t keys_bytes = exchange_keys_bytes(X.max_rows, X.world);
    const long long nblocks = exchange_blocks(X.max_rows);
    if (has_row) {
        for (int p = 0; p < X.world; ++p) {
            unsigned long long* dst = reinterpret_cast<unsigned long long*>(X.peer[p]) +
                                      ((size_t)parity * X.world + X.rank) * slot_keys + r * 2;
            *reinterpret_cast<ulonglong2*>(dst) = mine;
        }
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x < X.world) {
        const int p = threadIdx.x;
        unsigned* flag = reinterpret_cast<unsigned*>(X.peer[p] + keys_bytes) + (size_t)X.rank * nblocks + block;
        st_release_sys(flag, X.epoch);
        const unsigned* want = reinterpret_cast<const unsigned*>(X.peer[X.rank] + keys_bytes) + (size_t)p * nblocks + block;
        unsigned spins = 0;
        while ((int)(ld_acquire_sys(want) - X.epoch) < 0) {
            if (++spins > (1u << 27)) __trap();          // a missing peer must not hang the GPU
        }
    }
    __syncthreads();
    unsigned long long k1 = kNoMatch, k2 = kNoMatch;
    if (has_row) {
        const unsigned long long* base = reinterpret_cast<const unsigned long long*>(X.peer[X.rank]) +
                                         (size_t)parity * X.world * slot_keys + r * 2;
        for (int g = 0; g < X.world; ++g) {
            ulonglong2 k = mine;
            if (g != X.rank) {   // written by a peer GPU: bypass L1
                asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];\n"
                             : "=l"(k.x), "=l"(k.y)
                             : "l"(base + (size_t)g * slot_keys)
                             : "memory");
            }
            top2_insert(k1, k2, k.x);
            top2_insert(k1, k2, k.y);
        }
    }
    return make_ulonglong2(k1, k2);
}

inline size_t counters_bytes(long long row_blocks) { return (size_t)((row_blocks * 4 + 255) / 256 * 256); }

// ---- launchers implemented in the .cu files -------------------------------------------
// (a) POPC variant.  partial == nullptr -> writes final keys to out.
int popc_splits(const KnnProblem& p, int sm_count);
int launch_popc_knn2(const KnnProblem& p, unsigned long long* out, void* ws, size_t ws_bytes,
                     int sm_count, cudaStream_t stream);
size_t popc_workspace_bytes(long long nq, long long nt, int batch, int sm_count);

// (b) tensor-core variants (hm_tc.cu); `variant` is HM_VARIANT_I8 or HM_VARIANT_F4.
size_t prepared_bytes(long long n, int variant);
int launch_prepare(const uint8_t* bits, long long n, long long stride, long long batch_stride, int batch,
                   void* prepared, int variant, cudaStream_t stream);
// out == nullptr: leave the per-split partials in the workspace and report them through
// out_partials / out_groups instead of merging
int launch_tc_knn2_prepared(const void* qprep, long long nq, const void* tprep, long long nt, int batch,
                            unsigned long long train_base, unsigned long long* out, void* ws,
                            size_t ws_bytes, int sm_count, int variant, cudaStream_t stream,
                            const unsigned long long** out_partials = nullptr, int* out_groups = nullptr,
                            const ExchangeArgs* exchange = nullptr);
size_t tc_resident_workspace_bytes(long long nq, long long nt, int sm_count, int variant);
int launch_tc_knn2_resident(const uint8_t* qbits, long long nq, long long q_stride, const void* tprep, long long nt,
                            unsigned long long train_base, unsigned long long* out, void* ws, size_t ws_bytes,
                            int sm_count, int variant, cudaStream_t stream, const ExchangeArgs* exchange = nullptr);
int fill_exchange_args(ExchangeArgs* x, int world, int rank, void* const* peers, long long max_rows, unsigned epoch,
                       long long rows);
// the same over the selected runs of the prepared rows only; `totals` from the host copy of the runs (workspace:
// tc_resident_workspace_bytes(nq, totals.tiles * 128, ...))
int launch_tc_knn2_resident_runs(const uint8_t* qbits, long long nq, long long q_stride, const void* tprep, long long nt,
                                 const RunArgs& runs, const RunTotals& totals, unsigned long long train_base,
                                 unsigned long long* out, void* ws, size_t ws_bytes, int sm_count, int variant,
                                 cudaStream_t stream, const ExchangeArgs* exchange = nullptr);
// the physical tile sequence the CTAs of a run launch walk: out[v] = (split, tile, first column, end column) for
// virtual tile v, columns shard-local and clipped to the run (host arithmetic, the kernel's own walk)
void describe_tc_runs(long long nq, const long long* runs_host4, int n_runs, long long tiles, int sm_count, int variant,
                      char* buf, size_t n, long long* pieces);
size_t tc_workspace_bytes(long long nq, long long nt, int batch, int sm_count, bool with_prepare, int variant);
int launch_tc_knn2(const KnnProblem& p, unsigned long long* out, void* ws, size_t ws_bytes, int sm_count,
                   int variant, cudaStream_t stream);
// kind::mxf4 only.  Top-1 of the train rows list[b][0 .. count[b]) (device-side list and count) against all query
// rows: out[b][slot] = best query of candidate `slot`.  p.q / p.nq = the TRAIN side (gathered), p.t / p.nt = the query
// side (prepared into the workspace, which must hold tc_workspace_bytes(p.nq, p.nt, ..., with_prepare)).
int launch_tc_knn1_candidates(const KnnProblem& p, const int* list, const int* count, unsigned long long* out, void* ws,
                              size_t ws_bytes, int sm_count, cudaStream_t stream);

// epilogues
int launch_merge_top2(const unsigned long long* keys, int groups, long long rows, unsigned long long* out,
                      cudaStream_t stream);

size_t exchange_bytes(long long max_rows, int world);
int launch_exchange_merge(const unsigned long long* local_keys, int local_groups, long long rows, int world, int rank,
                          void* const* peers, long long max_rows, unsigned epoch, unsigned long long* out,
                          cudaStream_t stream);

// slot_of != null: bwd holds one entry per CANDIDATE train row (SelectArgs), train row t at slot_of[t] - 1;
// mutual_flags != null: the mutual check reads mutual_flags[b][q] instead of bwd (keyframe database, hm_db_filter)
int launch_filter(const unsigned long long* fwd, long long nq, const unsigned long long* bwd, long long nt,
                  int batch, unsigned flags, const RatioLut& lut, int thr_ceil, int* out_q, int* out_t,
                  int* out_d, int* out_count, cudaStream_t stream, const int* slot_of = nullptr,
                  const unsigned char* mutual_flags = nullptr);

// keyframe-database mutual check, one shard (hm_db_mutual_flags).  select: flags[0 .. nq) = 0 and the ordered list of
// the queries whose best row lies in [row_lo, row_hi) (and pass the ratio test when use_ratio): list[s] = local shard
// row, owner[s] = query, *count = entries; with `gathered` != null also gathered[s] = the shard row's 32 bytes (rows
// past *count zeroed).  resolve: flags[owner[s]] = 1 iff best[s] (top-1 key over the queries) names owner[s].
int launch_db_select(const unsigned long long* keys, long long nq, unsigned long long row_lo, unsigned long long row_hi,
                     int use_ratio, const RatioLut& lut, const uint8_t* shard_bits, long long t_stride, int* list,
                     int* owner, int* count, uint8_t* gathered, unsigned char* flags, cudaStream_t stream);
int launch_db_resolve(const int* owner, const int* count, const unsigned long long* best, long long nq,
                      unsigned char* flags, cudaStream_t stream);

void describe_tc_launch(long long nq, long long nt, int batch, int sm_count, int variant, bool top1, char* buf, size_t n);
int launch_gather_points(const int* q_idx, const int* t_idx, const int* count, long long stride, int batch,
                         const int* query_pts, long long nq, const int* train_pts, long long nt, int* out_query,
                         int* out_train, cudaStream_t stream);

// single-launch small-problem pipeline (hm_small.cu)
bool small_match_eligible(long long nq, long long nt);
int launch_small_match(const uint8_t* q, long long nq, const uint8_t* t, long long nt, unsigned flags, const RatioLut& lut,
                       int thr_ceil, int* out_mapped, unsigned epoch, cudaStream_t stream);

// ORB descriptor stage (hm_orb.cu)
size_t orb_workspace_bytes(int rows, int cols, int n_levels);
int launch_orb_pyramid(const uint8_t* image, int rows, int cols, long long row_stride, int channels, int n_levels, void* ws,
                       size_t ws_bytes, cudaStream_t stream);
int launch_orb_describe(const void* ws, int rows, int cols, int n_levels, const float* xy, const float* cs, const int* octave,
                        long long n, uint8_t* out, long long out_stride, cudaStream_t stream);
void orb_angles_to_cs(const float* angle_deg, long long n, float* cs);

int launch_rasterize_mask(const int* pts, long long n, int radius, int inner, unsigned char* mask, int h, int w,
                          long long row_stride, cudaStream_t stream);

}  // namespace hm
