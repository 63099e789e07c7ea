// Tensor-core variants: a tcgen05 GEMM on the +/-1 expansion of the descriptors.
//
// dot(a, b) over the +/-1 images of two 256-bit descriptors is 256 - 2*H, so the exact Hamming
// distance is H = (256 - dot) / 2 and "nearest" is "largest dot".  Two cores share one kernel body:
//
//   (b)  kind::i8    +/-1 as int8, 256 B per descriptor, K = 32 elements per MMA, s32 accumulators
//                    (the variant the north star names);
//   (b') kind::mxf4  +/-1 as e2m1 4-bit floats (+1.0 = 0x2, -1.0 = 0xA), 128 B per descriptor, K = 64
//                    elements per MMA, every ue8m0 block scale = 1.0, fp32 accumulators.  The dot
//                    products are small integers, exact in fp32, and the instruction issues at twice
//                    the kind::i8 rate (tools/microbench_fp4.cu: 16381 vs 8191 MAC/clk/SM, one
//                    128x128x256 tile bit-exact incl. dot = +/-256) with half the operand bytes.
//
// One CTA owns 256 query rows (two 128-row A blocks, resident in shared memory) and streams 128-row
// train tiles (B operand) through a ring of bulk-async-copy stages.  Per (tile, query block) a single
// elected thread issues the MMAs (M=128, N=128) into one of the 128-column TMEM accumulator units;
// epilogue warps (kind::i8: eight, one per 32 query rows; kind::mxf4: sixteen, two column halves per
// lane quarter) read finished units with tcgen05.ld (thread = query row, registers = train columns) and
// keep the running top-2 in registers -- at the granularity of 8-column groups, see Top2 -- so the distance tile
// never leaves the SM.  kind::i8 uses four units (2 query blocks x 2 buffers = all 512 columns); kind::mxf4 rotates
// three units and keeps its scale factors in the last 32 columns; its CTA carries a fifth warpgroup that hands
// registers to the epilogue warps (setmaxnreg, see threads()).  Three kernels per core: top-2, top-2 with row thresholds shared
// by all CTAs of a query row (split launches), top-1 (passes whose second neighbour nobody reads).
//
// Why this shape (ncu, profiles/r01a_* .. r01g_*): the +/-1 operands are 8x (4x) larger than the
// packed bits, so with 128 query rows per CTA each tile needs 64 B/clk/SM of L2->SM traffic and two
// stages cannot cover the ~2500-cycle load latency.  256 query rows per CTA halve the bytes per MMA
// cycle and leave room for 128 KB in flight.  CTAs are launched as thread-block clusters of 2 query
// blocks that share every train tile: each CTA fetches 1/CS of the tile and multicasts it
// (cp.async.bulk ... .multicast::cluster), and a stage is released by the multicast tcgen05.commit
// of all CS MMA issuers.
//
// Replaces the same cv::batchDistance loop as hm_popc.cu
// (/root/reference/feature_matchers.py:39 -> cv2.BFMatcher).
//
// Operands are "prepared" once by hm_prepare(): rows grouped in blocks of 128, each block stored
// exactly as the UMMA K-major SWIZZLE_128B shared-memory image (128-byte K slabs: two per row block
// for int8, one for e2m1), so a train tile is ONE contiguous bulk copy with no tensor map.
#include <math.h>
#include <stdlib.h>

#include <mutex>
#include <type_traits>

#include <cuda_fp16.h>

#include "hm_common.cuh"
#include "hm_tcgen05.cuh"

namespace hm {

namespace {

constexpr int kRowBlock = 128;               // rows per prepared block = UMMA M = tile N
constexpr int kMBlocks = 2;                  // A blocks per CTA
constexpr int kBlockM = kRowBlock * kMBlocks;   // 256 queries per CTA
// train rows per tile = MMA N: a per-core constant (C::kTileN)
constexpr int kSlabBytes = kRowBlock * 128;  // 16 KB: 128 rows x 128 bytes of K
constexpr int kPadRows = HM_PREPARED_TILE_ROWS;
constexpr int kTmemCols = 512;
// 4 * kMBlocks * kColSplit epilogue warps (one per 32 query rows and per 128 / kColSplit columns of a tile), then
// the producer and the MMA issuer
constexpr uint32_t kSpinLimit = 1u << 26;

static_assert(kPadRows % kBlockM == 0, "prepared padding must cover whole query blocks");

// ---- the two cores ---------------------------------------------------------------------------
struct CoreI8 {
    using Acc = int;
    static constexpr int kSlabs = 2;                         // 128-byte K slabs per row
    static constexpr int kRowBytes = HM_PREPARED_ROW_BYTES;  // 256
    static constexpr int kTileN = 128;                       // train rows per tile (one prepared row block)
    static constexpr int kStages = 4;                        // 4 x 32 KB in flight
    static constexpr int kUnits = 4;                         // accumulator units of kTileN TMEM columns
    static constexpr int kColSplit = 1;                      // 8 epilogue warps: the MMA (and the power cap) paces this core
    static constexpr bool kRegisterHandover = false;         // 10 warps: 168 registers per thread as launched
    static constexpr bool kScales = false;
    static constexpr int kPrologueTiles = 45;                // fixed per-CTA cost in tile times (split planning; half the kind::mxf4 figure: its tiles last twice as long)
    static __device__ __forceinline__ Acc lowest() { return INT_MIN; }
    static __device__ __forceinline__ Acc from_bits(uint32_t x) { return (int)x; }
    static __device__ __forceinline__ Acc max3(Acc a, Acc b, Acc c) { return __vimax3_s32(a, b, c); }
    static __device__ __forceinline__ Acc max2(Acc a, Acc b) { return max(a, b); }
    static __device__ __forceinline__ bool valid(Acc v) { return v >= -256; }
    static __device__ __forceinline__ unsigned distance(Acc v) { return (unsigned)((256 - v) >> 1); }
    static __device__ __forceinline__ unsigned encode(Acc v) { return (unsigned)(v + 257); }          // 1..513, 0 = none
    static __device__ __forceinline__ Acc floor_from(unsigned e) { return (int)e - 259; }             // dot - 2
    // two dots (|dot| <= 256, or the "no column" marker) in one register: the saved values of a candidate group
    static __device__ __forceinline__ uint32_t pack2(uint32_t lo, uint32_t hi) { return ((uint32_t)max((int)lo, -32768) & 0xFFFFu) | ((uint32_t)max((int)hi, -32768) << 16); }
    static __device__ __forceinline__ Acc unpack(uint32_t p, int hi) { return hi ? (int)p >> 16 : (int)(short)(p & 0xFFFFu); }
    static constexpr uint32_t kLowestBits = 0x80000000u;
};

struct CoreF4 {
    using Acc = float;
    static constexpr int kSlabs = 1;
    static constexpr int kRowBytes = HM_PREPARED_F4_ROW_BYTES;  // 128
    // The e2m1 image is a flat sequence of 8-row swizzle atoms, so any tile height that is a multiple of 8 is
    // one contiguous bulk copy.  96-row tiles let FOUR accumulator units fit beside the scale factors
    // (4 x 96 = 384 columns) and were tried to give the issuer more slack when an epilogue warp takes the
    // exact-insertion path: bit-exact, but 903 instead of 785 cycles per 128 columns on C4 (per-tile costs of
    // the issuer and of the epilogue warps do not shrink with the tile) -- so 128 rows and three units.
    static constexpr int kTileN = 128;
    // x 16 KB in flight.  Six stages (a multiple of the three accumulator units) keep the issuer's unrolled
    // period at six tiles; 96 KB cover > 4000 cycles of tile time against ~2500 cycles of load latency.
    static constexpr int kStages = 6;
    // accumulator units of kTileN columns in [0, 480); the scale factors live in the last 32 columns
    static constexpr int kUnits = 3;
    // 16 epilogue warps, two per (query block, lane quarter), 64 columns each: with 8 the scan is latency
    // bound (ncu r01j: issue slots 37 %, ALU 46 %, top stalls wait / long scoreboard) at 1087 cycles per
    // tile while the MMAs need 512
    static constexpr int kColSplit = 2;
    static constexpr bool kRegisterHandover = true;
    static constexpr bool kScales = true;
    // fixed cost of a CTA in steady-state tile times: launch + pipeline fill, the branch-free first tiles and the
    // slow early tiles before the thresholds settle.  Measured (2000 queries, 512 k ... 8.19 M train rows, DESIGN.md):
    // time per CTA = ~55-70 k cycles + 655 cycles per tile, i.e. 85-105 tiles -- not the 10 that were guessed before
    static constexpr int kPrologueTiles = 90;
    static __device__ __forceinline__ Acc lowest() { return -INFINITY; }
    static __device__ __forceinline__ Acc from_bits(uint32_t x) { return __uint_as_float(x); }
    static __device__ __forceinline__ Acc max3(Acc a, Acc b, Acc c) { return fmaxf(fmaxf(a, b), c); }   // FMNMX3
    static __device__ __forceinline__ Acc max2(Acc a, Acc b) { return fmaxf(a, b); }
    static __device__ __forceinline__ bool valid(Acc v) { return v >= -256.0f; }
    static __device__ __forceinline__ unsigned distance(Acc v) { return (unsigned)((256 - (int)v) >> 1); }
    static __device__ __forceinline__ unsigned encode(Acc v) { return (unsigned)((int)v + 257); }
    static __device__ __forceinline__ Acc floor_from(unsigned e) { return (float)((int)e - 259); }
    // f16x2: exact for integers up to 2048, and -inf stays -inf; one F2FP per pair
    static __device__ __forceinline__ uint32_t pack2(uint32_t lo, uint32_t hi)
    {
        const __half2 h = __floats2half2_rn(__uint_as_float(lo), __uint_as_float(hi));
        return *reinterpret_cast<const uint32_t*>(&h);
    }
    static __device__ __forceinline__ Acc unpack(uint32_t p, int hi)
    {
        const __half2 h = *reinterpret_cast<const __half2*>(&p);
        return hi ? __high2float(h) : __low2float(h);
    }
    static constexpr uint32_t kLowestBits = 0xFF800000u;
};

template <class C> __host__ __device__ constexpr int row_block_bytes() { return kRowBlock * C::kRowBytes; }
template <class C> __host__ __device__ constexpr int a_bytes() { return kMBlocks * row_block_bytes<C>(); }
template <class C> __host__ __device__ constexpr int b_stage_bytes() { return C::kTileN * C::kRowBytes; }
template <class C> __host__ __device__ constexpr int epilogue_warps() { return 4 * kMBlocks * C::kColSplit; }
// kind::mxf4: 16 epilogue warps + producer + issuer = 18 warps put five warps on two of the four SM sub-partitions, which
// caps every thread at 96 registers (16384 / (5 * 32) rounded down to 8).  The CTA is therefore launched with a full
// fifth warpgroup -- producer, issuer and two idle warps -- that hands registers to the epilogue warps at entry
// (setmaxnreg: 4 x 32 + 16 x 112 = 20 x 96 registers per thread-slot): the scan keeps 64 accumulator values, the
// running top-2 and the saved dots of two candidate groups in registers without spilling.
template <class C> __host__ __device__ constexpr int control_warps() { return C::kRegisterHandover ? 4 : 2; }
template <class C> __host__ __device__ constexpr int threads() { return 32 * (control_warps<C>() + epilogue_warps<C>()); }
// + 256 B of barriers, + 4 KB where the epilogue warps of the upper column halves hand over their keys
constexpr int kHandoverBytes = kBlockM * 16;
constexpr int kBarrierBytes = 512;
template <class C> __host__ __device__ constexpr int smem_bytes() { return 1024 + a_bytes<C>() + C::kStages * b_stage_bytes<C>() + kBarrierBytes + kHandoverBytes; }
static_assert((2 * CoreF4::kStages + 1 + 2 * CoreF4::kUnits) * 8 + 16 <= kBarrierBytes, "barrier block");
static_assert((2 * CoreI8::kStages + 1 + 2 * CoreI8::kUnits) * 8 + 16 <= kBarrierBytes, "barrier block");
__host__ __device__ constexpr int ct_gcd(int a, int b) { return b == 0 ? a : ct_gcd(b, a % b); }
// tiles after which the stage ring AND the accumulator-unit rotation (two items per tile) are back where they started
template <class C> __host__ __device__ constexpr int issuer_period() { return C::kStages / ct_gcd(C::kStages, C::kUnits) * C::kUnits; }
// Scale factors: one 32-bit TMEM cell holds four ue8m0 bytes; an M = 128 (N = 128) operand needs 4 columns of them.
// Every scale is 1.0 (0x7F), so the layout inside the region does not matter: the last 32 columns are filled once,
// A reads its scales at column 480, B at 496.
constexpr int kScaleCols = 32;
constexpr int kScaleCol = kTmemCols - kScaleCols;
static_assert(CoreF4::kUnits * CoreF4::kTileN <= kScaleCol, "accumulator units must end before the scale factors");

// ---- run walk (hm_knn2_resident_runs) ------------------------------------------------------------
// A selection of rows is a list of ascending, disjoint runs [lo, hi) (RunArgs).  Its virtual tiles [0, T) are the
// 128-row tiles each run touches, run after run: a tile two runs share (across a short unselected stretch) appears
// once per run, the lower run first.  Split s of a launch takes virtual tiles [s * tiles_per_split, ...).  The kernel's
// producer and epilogue warps and describe_tc_runs walk the same sequence with this cursor.
struct RunCursor {
    int r;                       // current run
    int tile, end;               // physical tile; one past the run's last tile
    unsigned lo, hi;             // the run's rows (shard-local): columns outside [lo, hi) must never win
    __host__ __device__ __forceinline__ void load(const long long* runs, int rr)
    {
        r = rr;
        const long long a = runs[kRunFields * rr], b = runs[kRunFields * rr + 1];
        lo = (unsigned)a;
        hi = (unsigned)b;
        tile = (int)(a / kRowBlock);
        end = (int)((b + kRowBlock - 1) / kRowBlock);
    }
    // position at virtual tile v: the last run whose tile prefix is <= v (prefixes strictly increase: runs are non-empty)
    __host__ __device__ __forceinline__ void seek(const long long* runs, int n_runs, long long v)
    {
        int a = 0, b = n_runs - 1;
        while (a < b) {
            const int m = (a + b + 1) >> 1;
            if (runs[kRunFields * m + 2] <= v) a = m;
            else b = m - 1;
        }
        load(runs, a);
        tile += (int)(v - runs[kRunFields * a + 2]);
    }
    // the next virtual tile; only called when there is one
    __host__ __device__ __forceinline__ void next(const long long* runs)
    {
        if (++tile == end) load(runs, r + 1);
    }
};
static_assert(CoreI8::kTileN == kRowBlock && CoreF4::kTileN == kRowBlock, "the run walk counts tiles of kRowBlock rows");

// ------------------------------------------------------------------------------------------
// hm_prepare: packed bits -> +/-1 in the tiled swizzled layout.  One thread writes one 16-byte
// chunk (16 descriptor bits as int8, 32 as e2m1); consecutive threads write consecutive chunks.
// ------------------------------------------------------------------------------------------
struct PrepareParams {
    const uint8_t* bits;
    long long n, stride, batch_stride;
    long long padded_rows;
    uint8_t* out;
};

__global__ void __launch_bounds__(256) hm_prepare_kernel(const PrepareParams P)
{
    const long long chunks_per_problem = P.padded_rows * 16;
    const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= chunks_per_problem) return;
    const int b = blockIdx.y;
    const long long rb = o >> 11;            // 2048 chunks per 128-row block
    const int rem = (int)(o & 2047);
    const int slab = rem >> 10;
    const int rem2 = rem & 1023;
    const int rr = (rem2 >> 3) & 7;          // row within its 8-row group
    const int r = ((rem2 >> 6) << 3) | rr;   // row within the block
    const int c = (rem2 & 7) ^ rr;           // logical 16-byte chunk stored at this position
    const long long row = rb * kRowBlock + r;
    uint4 v = make_uint4(0, 0, 0, 0);        // padding rows stay zero
    if (row < P.n) {
        const uint8_t* src = P.bits + (long long)b * P.batch_stride + row * P.stride + slab * 16 + c * 2;
        const unsigned bits16 = (unsigned)src[0] | ((unsigned)src[1] << 8);
        unsigned w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const unsigned nib = (bits16 >> (4 * i)) & 0xF;
            const unsigned spread = (nib & 1) | ((nib & 2) << 7) | ((nib & 4) << 14) | ((nib & 8) << 21);
            w[i] = (spread * 0xFEu) ^ 0xFFFFFFFFu;   // bit 1 -> 0x01 (+1), bit 0 -> 0xFF (-1)
        }
        v = make_uint4(w[0], w[1], w[2], w[3]);
    }
    uint4* dst = reinterpret_cast<uint4*>(P.out + (long long)b * P.padded_rows * HM_PREPARED_ROW_BYTES);
    dst[o] = v;
}

// 32 descriptor bits -> 32 e2m1 values (16 bytes): bit j -> nibble j, set = +1.0 (0x2), clear = -1.0 (0xA)
__device__ __forceinline__ uint4 expand_bits_e2m1(unsigned bits32)
{
    unsigned w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const unsigned by = (bits32 >> (8 * i)) & 0xFF;
        unsigned sgn = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) sgn |= ((by >> j) & 1u) << (4 * j + 3);
        w[i] = 0xAAAAAAAAu ^ sgn;
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}

// e2m1 image: one 128-byte slab per row, chunk c = descriptor bytes [4c, 4c+4)
__global__ void __launch_bounds__(256) hm_prepare_f4_kernel(const PrepareParams P)
{
    const long long chunks_per_problem = P.padded_rows * 8;
    const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= chunks_per_problem) return;
    const int b = blockIdx.y;
    const long long rb = o >> 10;            // 1024 chunks per 128-row block
    const int rem = (int)(o & 1023);
    const int rr = (rem >> 3) & 7;
    const int r = ((rem >> 6) << 3) | rr;
    const int c = (rem & 7) ^ rr;
    const long long row = rb * kRowBlock + r;
    uint4 v = make_uint4(0, 0, 0, 0);        // padding rows: +0.0 everywhere
    if (row < P.n) {
        const unsigned bits32 = *reinterpret_cast<const unsigned*>(P.bits + (long long)b * P.batch_stride + row * P.stride + c * 4);
        v = expand_bits_e2m1(bits32);
    }
    uint4* dst = reinterpret_cast<uint4*>(P.out + (long long)b * P.padded_rows * HM_PREPARED_F4_ROW_BYTES);
    dst[o] = v;
}

// ------------------------------------------------------------------------------------------
// main kernel
// ------------------------------------------------------------------------------------------
struct TcParams {
    // kind::mxf4 only: packed query descriptors.  When set, every CTA expands its 256 query rows into the A operand
    // image in shared memory itself (8 KB of bits -> 32 KB of e2m1) and `qprep` is not read: no hm_prepare launch
    // for the query side, one launch per k-NN call.
    const uint8_t* qbits;
    long long q_bits_stride, q_bits_batch_stride;
    // with qbits: query row r of problem b is row q_index[b * q_index_batch_stride + r] of the packed array (a gather
    // folded into the expansion), and only the first nq_dyn[b] (<= nq) query rows exist -- a row count produced on the
    // device by an earlier kernel of the same stream.  Clusters whose query blocks lie beyond it return at once.
    // This is the swapped pass of the mutual check restricted to the candidate train rows (hm_match_fused).
    const int* q_index;
    long long q_index_batch_stride;
    const int* nq_dyn;
    const uint8_t* qprep;            // [batch][q_padded][row bytes]
    const uint8_t* tprep;            // [batch][t_padded][row bytes]
    long long nq, nt;
    long long q_padded, t_padded;
    int tiles_per_split;             // train tiles (128 rows) per split
    int ntiles;                      // total train tiles
    unsigned long long train_base;
    unsigned long long* out;         // [split][batch][nq][2]
    long long out_split_stride;      // keys
    int* error_flag;
    unsigned long long* final_out;   // [batch][nq][2]: written by the last CTA of each query block when merging in-kernel
    unsigned* counters;              // [batch][qblocks] arrival counters (zeroed by the launcher), null = no in-kernel merge
    int splits;
    // [batch][nq] shared row thresholds (zeroed by the launcher), null = off.  Every CTA starts with an empty
    // top-2, so for its first ~40 tiles the scan's exact-insertion path runs for most chunks; with the train
    // set split over many CTAs per query row that warm-up dominated short CTAs (C3, C5, 8-GPU shards).  The
    // CTAs of a row therefore publish the second-best dot they have found (atomicMax on a monotone code)
    // and read the row's value back every few tiles: any published value is a lower bound of the row's final
    // second best, so columns strictly below it are skipped without touching the result.
    unsigned* row_floor;
    ExchangeArgs xch;                // xch.world > 1: the last CTA also exchanges with the peer GPUs (sharded database)
    long long q_blocks_valid;        // 256-row blocks present in qprep (CTAs beyond it are cluster padding)
    // [4] measurement aid, always on (one thread, four stores): %globaltimer (ns) and clock64 (SM cycles) of CTA
    // (0,0,0) at entry and exit.  Their ratio is the SM clock actually running under this kernel -- NVML, polled every
    // few ms, keeps reporting the 1965 MHz application clock while the chip runs the tensor pipe at ~1.65-1.75 GHz.
    long long* clock_probe;
    SelectArgs sel;                  // sel.slot_of != null: ratio test + candidate-column selection on the final keys
};

// Running top-2 of one query row at GROUP granularity.  A group is 8 consecutive train columns.  The scan keeps the
// two groups with the largest maxima (earliest group on ties) and a copy of their 8 dots each, packed two per
// register; the exact (distance, trainIdx) top-2 is taken from those 16 saved dots once, at the end of the CTA.
// Why that is exact: the best column (largest dot, lowest index) lies in the earliest group whose maximum is the
// overall maximum = g1.  Any group other than g1 and g2 has a maximum <= v2 and, on equality, a later position than
// g2, so each of its columns loses against g1's best AND against g2's best: the second-best column lies in g1 or g2.
// What this buys: a candidate costs one compare per GROUP and ~15 predicated instructions for the group that holds
// it, instead of a compare-and-insert chain over its 8 columns -- the path every warp is on while the thresholds are
// still low (CTAs that see fewer than ~10^4 columns: C2, C3, C5, 8-GPU shards never leave it).
template <class Acc>
struct Top2 {
    Acc v1, v2;                      // largest / second-largest group maximum (larger dot = closer)
    unsigned i1, i2;                 // first column of those groups, local to this CTA's range
    uint32_t sa[4], sb[4];           // their 8 dots (C::pack2)
    // Filter threshold f = max(v2, shared) where `shared` = (second-best dot some CTA of this row has already
    // published, see TcParams::row_floor) - 2.  A group can only matter if its maximum is > v2 (to enter the local
    // top-2) and >= the published second best (to enter the row's final top-2; dots are even, so "> shared"):
    // one compare against f skips everything else.  v2 only grows, so after an insertion
    // max(v2_new, shared) = max(v2_new, f_old) and `shared` itself need not be kept.
    Acc f;
};

__device__ __forceinline__ void bounded_wait(uint64_t* bar, uint32_t parity, int* error_flag)
{
    uint32_t spins = 0;
    while (!ptx::mbar_try_wait(bar, parity)) {
        if (++spins > kSpinLimit) {          // a protocol bug must not hang the GPU
            if (error_flag) atomicExch(error_flag, 1);
            __trap();
        }
    }
}

__device__ __forceinline__ void bounded_wait_addr(uint32_t bar_addr, uint32_t parity, int* error_flag)
{
    uint32_t spins = 0;
    while (!ptx::mbar_try_wait_addr(bar_addr, parity)) {
        if (++spins > kSpinLimit) {
            if (error_flag) atomicExch(error_flag, 1);
            __trap();
        }
    }
}

#define HM_R8(a, o) "+r"(a[o]), "+r"(a[o + 1]), "+r"(a[o + 2]), "+r"(a[o + 3]), "+r"(a[o + 4]), "+r"(a[o + 5]), "+r"(a[o + 6]), "+r"(a[o + 7])
#define HM_R32(a) HM_R8(a, 0), HM_R8(a, 8), HM_R8(a, 16), HM_R8(a, 24)
// one wait for four outstanding 32-column loads (128 registers pinned behind it)
__device__ __forceinline__ void tmem_ld_fence4(uint32_t (&a)[32], uint32_t (&b)[32], uint32_t (&c)[32], uint32_t (&d)[32])
{
    asm volatile("tcgen05.wait::ld.sync.aligned;\n" : HM_R32(a), HM_R32(b), HM_R32(c), HM_R32(d) : : "memory");
}
__device__ __forceinline__ void tmem_ld_fence64(uint32_t (&a)[64])
{
    asm volatile("tcgen05.wait::ld.sync.aligned;\n" : HM_R8(a, 0), HM_R8(a, 8), HM_R8(a, 16), HM_R8(a, 24), HM_R8(a, 32), HM_R8(a, 40), HM_R8(a, 48), HM_R8(a, 56) : : "memory");
}

// 32 (64) consecutive train columns of one query row.  Fast path: 3-input-max trees give the maximum of each group
// of 8 columns and of the whole chunk; one compare + branch per chunk against the threshold decides whether anything
// can change the top-2.  Only then are the group maxima revisited; a group above the threshold is inserted into the
// top-2 of groups together with a packed copy of its dots.  Strict '>' in ascending column order keeps the earliest
// group on ties, which is what the lowest-trainIdx rule needs (see Top2).
// kMode: 0 = top-2, 1 = top-2 with the shared row threshold, 2 = top-1 only (the swapped pass of the mutual
// check needs nothing else: the threshold is then the best dot itself, so the insertion path fires about half as
// often)
template <class C, int kMode, int kGroups = 4>
__device__ __forceinline__ void scan_chunk(const uint32_t* r, unsigned colbase, Top2<typename C::Acc>& s)
{
    using Acc = typename C::Acc;
    static_assert(kGroups == 4 || kGroups == 8, "8-column groups per compare");
    Acc gm[kGroups];
#pragma unroll
    for (int g = 0; g < kGroups; ++g) {
        const int o = g * 8;
        gm[g] = C::max3(C::max3(C::from_bits(r[o]), C::from_bits(r[o + 1]), C::from_bits(r[o + 2])),
                        C::max3(C::from_bits(r[o + 3]), C::from_bits(r[o + 4]), C::from_bits(r[o + 5])),
                        C::max2(C::from_bits(r[o + 6]), C::from_bits(r[o + 7])));
    }
    Acc m;
    if constexpr (kGroups == 8) m = C::max3(C::max3(gm[0], gm[1], gm[2]), C::max3(gm[3], gm[4], gm[5]), C::max2(gm[6], gm[7]));
    else m = C::max3(gm[0], gm[1], C::max2(gm[2], gm[3]));
    constexpr bool kFloor = kMode == 1, kTop1 = kMode == 2;
    if (m > (kFloor ? s.f : kTop1 ? s.v1 : s.v2)) {
#pragma unroll
        for (int g = 0; g < kGroups; ++g) {
            const Acc x = gm[g];
            if (x > (kFloor ? s.f : kTop1 ? s.v1 : s.v2)) {
                const int o = g * 8;
                const uint32_t p0 = C::pack2(r[o], r[o + 1]), p1 = C::pack2(r[o + 2], r[o + 3]);
                const uint32_t p2 = C::pack2(r[o + 4], r[o + 5]), p3 = C::pack2(r[o + 6], r[o + 7]);
                const unsigned idx = colbase + o;
                if (kTop1 || x > s.v1) {
                    if (!kTop1) {
                        s.v2 = s.v1; s.i2 = s.i1;
                        s.sb[0] = s.sa[0]; s.sb[1] = s.sa[1]; s.sb[2] = s.sa[2]; s.sb[3] = s.sa[3];
                    }
                    s.v1 = x; s.i1 = idx;
                    s.sa[0] = p0; s.sa[1] = p1; s.sa[2] = p2; s.sa[3] = p3;
                } else {
                    s.v2 = x; s.i2 = idx;
                    s.sb[0] = p0; s.sb[1] = p1; s.sb[2] = p2; s.sb[3] = p3;
                }
                if (kFloor) s.f = C::max2(s.v2, s.f);
            }
        }
    }
}

// columns at or beyond `limit` (the padding rows of the last train tile are +0.0: dot 0) must never win
template <class C, int kN>
__device__ __forceinline__ void mask_tail(uint32_t* r, unsigned colbase, unsigned limit)
{
    if (colbase + kN > limit) {
#pragma unroll
        for (int j = 0; j < kN; ++j)
            if (colbase + j >= limit) r[j] = C::kLowestBits;
    }
}

// run walk: columns outside the current run [lo, hi) -- in the run's first and last tile only -- must never win
template <class C, int kN>
__device__ __forceinline__ void mask_outside(uint32_t* r, unsigned colbase, unsigned lo, unsigned hi)
{
#pragma unroll
    for (int j = 0; j < kN; ++j)
        if (colbase + j < lo || colbase + j >= hi) r[j] = C::kLowestBits;
}

// the shared row thresholds are refreshed on each of a CTA's first kFloorDenseTiles tiles, then on every 16th
constexpr int kFloorDenseTiles = 32;
constexpr int kFloorLateMask = 15;

// half `h` (0 / 1) of the MMAs of one (tile, query block) item: kSlabs * 2 instructions
template <class C>
__device__ __forceinline__ void issue_half(int h, uint32_t a_block, uint32_t b_stage, uint32_t tmem_d, uint32_t idesc,
                                           uint32_t tmem_sf)
{
    constexpr int kHalf = C::kSlabs * 2;
#pragma unroll
    for (int jj = 0; jj < kHalf; ++jj) {
        const int j = h * kHalf + jj;
        const int slab = j >> 2, k = j & 3;
        // a_block / b_stage are descriptor start-address fields (shared-memory address >> 4)
        const uint64_t db = ptx::kmajor_sw128_desc_from_lo(b_stage + ((slab * kSlabBytes + k * 32) >> 4));
        const uint64_t da = ptx::kmajor_sw128_desc_from_lo(a_block + ((slab * kSlabBytes + k * 32) >> 4));
        if constexpr (C::kScales) ptx::mma_mxf4_ss(tmem_d, da, db, idesc, tmem_sf, tmem_sf + kScaleCols / 2, j != 0);
        else                      ptx::mma_i8_ss(tmem_d, da, db, idesc, j != 0);
    }
}

// kRuns: the train tiles come from the run list R (RunCursor) instead of tile_begin + i; columns are physical
// (shard-local rows, first_row = 0), so the final fold needs no remapping
template <class C, int kMode, bool kRuns = false>
__device__ __forceinline__ void tc_knn2_body(const TcParams& P, const RunArgs& R = RunArgs{})
{
    constexpr bool kFloor = kMode == 1;
    using Acc = typename C::Acc;
    constexpr int kStages = C::kStages;
    constexpr int kUnits = C::kUnits;
    constexpr int kABytes = a_bytes<C>();
    constexpr int kBStageBytes = b_stage_bytes<C>();
    constexpr int kRowBlockBytes = row_block_bytes<C>();
    constexpr int kTileN = C::kTileN;

    extern __shared__ uint8_t smem_raw[];
    // SWIZZLE_128B atoms need 1024-byte alignment
    uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* smem_a = smem;                      // [query block 0][query block 1], each [slab 0 | slab 1 ...]
    uint8_t* smem_b = smem + kABytes;            // kStages x one 128-row train tile
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kABytes + kStages * kBStageBytes);
    uint64_t* full_bar = bars;                   // [kStages]  bulk copies landed
    uint64_t* empty_bar = bars + kStages;        // [kStages]  MMAs reading the stage retired
    uint64_t* a_full_bar = bars + 2 * kStages;   // [1]
    // accumulator units of 128 TMEM columns; work item w = 2 * tile + query block uses unit w % kUnits
    uint64_t* tmem_full_bar = bars + 2 * kStages + 1;      // [kUnits] unit complete
    uint64_t* tmem_empty_bar = tmem_full_bar + kUnits;     // [kUnits] unit drained by its epilogue warps
    uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + kUnits);
    uint32_t* smem_base_slot = tmem_base_slot + 2;         // shared address of `smem` (see lds_volatile_u32)
    ulonglong2* handover = reinterpret_cast<ulonglong2*>(smem + kABytes + kStages * kBStageBytes + kBarrierBytes);   // [kBlockM]

    // broadcast from lane 0: lets ptxas treat the warp index (and the role branches on it) as warp-uniform
    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
    const int lane = threadIdx.x & 31;
    if (threadIdx.x == 0 && (blockIdx.x | blockIdx.y | blockIdx.z) == 0 && P.clock_probe) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        P.clock_probe[0] = (long long)t;
        P.clock_probe[1] = clock64();
    }
    const int qb = blockIdx.x;                   // 256-row query block
    const int split = blockIdx.y;
    const int b = blockIdx.z;

    const uint32_t cs = ptx::cluster_nctarank();            // 1, 2 or 4 CTAs sharing the B tiles
    const uint32_t crank = ptx::cluster_ctarank();
    const uint16_t cmask = (uint16_t)((1u << cs) - 1);
    const bool has_a = qb < P.q_blocks_valid;
    // query rows that exist: P.nq, or the device-side count of a candidate list (the stride of every per-row array
    // stays P.nq).  A cluster with no row left returns as a whole, before any barrier or TMEM allocation.
    // (re-evaluated where it is needed instead of being kept in registers across the tile loop)
    auto rows_present = [&]() -> long long { return P.nq_dyn ? min((long long)__ldg(P.nq_dyn + b), P.nq) : P.nq; };
    if (P.nq_dyn && (long long)(qb - (int)crank) * kBlockM >= rows_present()) return;

    const int tile_begin = split * P.tiles_per_split;
    const int tile_end = min(tile_begin + P.tiles_per_split, P.ntiles);
    const int my_tiles = tile_end - tile_begin;          // >= 1 by construction

    // Warp roles.  The SM sub-partition's arbiter issues the eligible warp with the HIGHEST index first
    // (/opt/skills/guides/B300_MICROARCH.md, "Multi-warp arbiter"), so the two latency-critical single warps -- the
    // MMA issuer above all -- are the LAST two warps of the CTA: the issuer never queues behind the four epilogue
    // warps that share its sub-partition.  Epilogue warps come first; warp % 4 is still their TMEM lane quarter.
    constexpr int kProducerWarp = epilogue_warps<C>();
    constexpr int kIssuerWarp = epilogue_warps<C>() + 1;
    static_assert(!C::kRegisterHandover || (epilogue_warps<C>() == 16 && threads<C>() == 640),
                  "the register budget (4 x 32 + 16 x 112 = 20 x 96) assumes 20 warps launched at 96 registers");
    if (warp == kProducerWarp && lane == 0) {
        *smem_base_slot = ptx::smem_u32(smem);
        for (int i = 0; i < kStages; ++i) {
            ptx::mbar_init(&full_bar[i], 1);
            ptx::mbar_init(&empty_bar[i], cs);           // one (multicast) commit per CTA of the cluster
        }
        ptx::mbar_init(a_full_bar, 1);
        for (int i = 0; i < kUnits; ++i) {
            ptx::mbar_init(&tmem_full_bar[i], 1);
            ptx::mbar_init(&tmem_empty_bar[i], 4 * C::kColSplit);   // one arrival per epilogue warp of the item's query block
        }
        ptx::fence_barrier_init();
        ptx::fence_proxy_async();
    } else if (warp == kIssuerWarp) {
        ptx::tmem_alloc(tmem_base_slot, kTmemCols);
        ptx::tmem_relinquish();
    }
    ptx::tc_fence_before();
    if (cs > 1) ptx::cluster_sync();   // peers' barriers are initialised before any multicast lands
    else __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_base_slot;

    if constexpr (C::kScales) {
        // every block scale is 1.0 (ue8m0 0x7F): fill the scale-factor columns once, all 128 lanes
        if ((unsigned)warp < 4) {          // the first four epilogue warps, one per lane quarter
            uint32_t ones[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) ones[i] = 0x7F7F7F7Fu;
            const uint32_t taddr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + kScaleCol;
            static_assert(kScaleCols == 32, "one x32 store per lane quarter");
            ptx::tmem_st_32x32(taddr, ones);
            ptx::tmem_st_wait();
        }
        if (P.qbits) {
            // A operand from packed bits: the same swizzled image hm_prepare_f4_kernel writes, straight into shared
            // memory (chunk position -> row and logical chunk as there); rows past nq are +0.0 like the padding
            const uint8_t* qsrc = P.qbits + (long long)b * P.q_bits_batch_stride;
            const int* qidx = P.q_index ? P.q_index + (long long)b * P.q_index_batch_stride : nullptr;
            const long long nq_eff = rows_present();
            for (int o = threadIdx.x; o < kBlockM * 8; o += blockDim.x) {
                const int blk = o >> 10, rem = o & 1023;
                const int rr = (rem >> 3) & 7;
                const int r = ((rem >> 6) << 3) | rr;
                const int c = (rem & 7) ^ rr;
                const long long qrow = (long long)qb * kBlockM + blk * kRowBlock + r;
                uint4 v = make_uint4(0, 0, 0, 0);
                if (qrow < nq_eff) {
                    const long long srow = qidx ? (long long)__ldg(qidx + qrow) : qrow;
                    v = expand_bits_e2m1(*reinterpret_cast<const unsigned*>(qsrc + srow * P.q_bits_stride + c * 4));
                }
                reinterpret_cast<uint4*>(smem_a)[o] = v;
            }
            ptx::fence_proxy_async();      // generic-proxy stores -> visible to the tensor core's async-proxy reads
        }
        ptx::tc_fence_before();
        __syncthreads();
        ptx::tc_fence_after();
    }

    ulonglong2 my_keys = make_ulonglong2(kNoMatch, kNoMatch);   // epilogue threads: top-2 keys of their row (and column half)
    long long my_row = -1;                                      // >= 0: this thread writes the row's keys
    int my_row_in_cta = 0;

    // The three roles and the common tail are lambdas so that the kind::mxf4 core can run the control warpgroup and the
    // epilogue warps as two separate straight-line paths with different register budgets (see the dispatch below).
    auto run_producer = [&]() {
        // ===== producer: bulk async copies global -> shared =====
        if (lane == 0) {
            if (has_a && !P.qbits) {
                const uint8_t* qsrc = P.qprep + ((long long)b * P.q_padded + (long long)qb * kBlockM) * C::kRowBytes;
                ptx::mbar_arrive_expect_tx(a_full_bar, kABytes);
                ptx::bulk_g2s(smem_a, qsrc, kABytes, a_full_bar);       // two consecutive row blocks
            }
            const uint8_t* tsrc = P.tprep + (long long)b * P.t_padded * C::kRowBytes;
            const uint32_t piece = kBStageBytes / cs;     // this CTA fetches 1/cs of every tile and multicasts it
            RunCursor cur;
            if constexpr (kRuns) cur.seek(R.runs, R.n_runs, tile_begin);
            for (int i = 0; i < my_tiles; ++i) {
                const int stage = i % kStages;
                const uint32_t use = i / kStages;
                bounded_wait(&empty_bar[stage], (use & 1) ^ 1, P.error_flag);
                ptx::mbar_arrive_expect_tx(&full_bar[stage], kBStageBytes);
                uint8_t* dst = smem_b + stage * kBStageBytes + crank * piece;
                int tile = tile_begin + i;
                if constexpr (kRuns) {
                    tile = cur.tile;
                    if (i + 1 < my_tiles) cur.next(R.runs);
                }
                const uint8_t* src = tsrc + (long long)tile * kBStageBytes + crank * piece;
                if (cs > 1) ptx::bulk_g2s_multicast(dst, src, piece, &full_bar[stage], cmask);
                else        ptx::bulk_g2s(dst, src, piece, &full_bar[stage]);
            }
        }
    };
    auto run_issuer = [&]() {
        // ===== MMA issuer =====
        // tcgen05.mma issue blocks while the tensor-core queue is full, so every barrier round trip
        // (~100-150 cycles) taken between two groups of MMAs is a bubble in the tensor pipe.  The
        // barriers of the NEXT group are therefore probed (mbarrier.test_wait, non-blocking) in the
        // middle of the current group, while its MMAs execute; the blocking wait is only the fallback.
        // The whole warp runs the loop so that counters, stage / unit indices, barrier addresses and the
        // shared-memory descriptors stay in the uniform datapath; only the tcgen05 instructions are
        // predicated on the elected lane.  (With the loop inside `if (elect_one())` every operand went
        // through a vector register and an R2UR: ~140 dependent instructions of one thread per tile, which
        // paced the kind::mxf4 core at 114 cycles per MMA instead of 64 -- profiles/r01k_trace_f4_c4_tiles1200.txt.
        // Two issuer warps (one per query block, per-(unit, block) barriers, stage released by an epilogue
        // thread) were tried twice: with the epilogue switched off they lower the floor from 622 to 557
        // cycles per tile, but with the real epilogue the kind::mxf4 core is slower (860-880 vs 803): the
        // items of both blocks then complete together, and three accumulator units cannot hide the
        // drain latency.  Also measured: an epilogue-driven stage release through
        // mbarrier.arrive.release.cluster costs the arriving thread ~2000 cycles per call (relaxed: none),
        // and blocking waits instead of the probes cost 70 cycles per tile.)
        const bool leader = ptx::elect_one();
        const uint32_t idesc = C::kScales ? ptx::make_mxf4_idesc(kRowBlock, kTileN) : ptx::make_i8_idesc(kRowBlock, kTileN);
        const uint32_t a_addr = ptx::smem_u32(smem_a) >> 4;       // descriptor start-address fields
        constexpr uint32_t kABlockStep = kRowBlockBytes >> 4;
        const uint32_t b_addr = ptx::smem_u32(smem_b) >> 4;
        const uint32_t tmem_sf = tmem_base + kScaleCol;
        if (has_a && !P.qbits) bounded_wait(a_full_bar, 0, P.error_flag);
        // The loop is unrolled over one period of the stage ring and of the unit rotation (kPeriod tiles), so that the
        // stage, the accumulator units, every barrier address, every descriptor offset and the unit parities are
        // compile-time constants: what is left per tile is the eight (sixteen) MMAs, three commits, the probes / waits
        // and the constant adds that build the descriptors.  (The rolled loop spent ~110 uniform-datapath
        // instructions per tile on index arithmetic, ~5 cycles each on the one issuing warp: 622 cycles per tile
        // even with the epilogue switched off, against 512 cycles of MMA.)
        constexpr int kPeriod = issuer_period<C>();
        static_assert(kPeriod % kStages == 0 && (2 * kPeriod) % kUnits == 0 && ((2 * kPeriod / kUnits) & 1) == 0,
                      "unit parities must repeat with the period");
        uint32_t sphase = 0;                          // parity of (tile / kStages) at the period's first tile
        bool ready0 = false;                          // full[stage] and empty[unit] of the next tile's first item observed
        for (int base = 0; base < my_tiles; base += kPeriod) {
#pragma unroll
            for (int j = 0; j < kPeriod; ++j) {
                if (base + j < my_tiles) {
                    const int stage = j % kStages;
                    const uint32_t full_par = sphase ^ ((j / kStages) & 1);
                    const int unit_a = (2 * j) % kUnits, unit_b = (2 * j + 1) % kUnits;
                    const uint32_t par_a = (((2 * j) / kUnits) & 1) ^ 1, par_b = (((2 * j + 1) / kUnits) & 1) ^ 1;
                    const uint32_t b_stage = b_addr + stage * (kBStageBytes >> 4);
                    if (!ready0) {
                        bounded_wait(&full_bar[stage], full_par, P.error_flag);
                        bounded_wait(&tmem_empty_bar[unit_a], par_a, P.error_flag);
                    }
                    ptx::tc_fence_after();
                    // ---- query block 0 ----
                    if (leader) issue_half<C>(0, a_addr, b_stage, tmem_base + unit_a * kTileN, idesc, tmem_sf);
                    const bool ready1 = __all_sync(0xffffffffu, ptx::mbar_test_wait(&tmem_empty_bar[unit_b], par_b));
                    if (leader) {
                        issue_half<C>(1, a_addr, b_stage, tmem_base + unit_a * kTileN, idesc, tmem_sf);
                        ptx::tc_commit(&tmem_full_bar[unit_a]);    // query block 0's accumulator is ready
                    }
                    // ---- query block 1 ----
                    if (!ready1) bounded_wait(&tmem_empty_bar[unit_b], par_b, P.error_flag);
                    ptx::tc_fence_after();
                    if (leader) issue_half<C>(0, a_addr + kABlockStep, b_stage, tmem_base + unit_b * kTileN, idesc, tmem_sf);
                    ready0 = false;
                    if (base + j + 1 < my_tiles) {
                        const int n = j + 1;                       // n == kPeriod wraps to stage 0 / unit 0 of the next period
                        ready0 = __all_sync(0xffffffffu,
                                            ptx::mbar_test_wait(&full_bar[n % kStages], sphase ^ ((n / kStages) & 1))
                                            && ptx::mbar_test_wait(&tmem_empty_bar[(2 * n) % kUnits], (((2 * n) / kUnits) & 1) ^ 1));
                    }
                    if (leader) {
                        issue_half<C>(1, a_addr + kABlockStep, b_stage, tmem_base + unit_b * kTileN, idesc, tmem_sf);
                        ptx::tc_commit(&tmem_full_bar[unit_b]);
                        // smem stage reusable (by every producer of the cluster) once these MMAs retire
                        if (cs > 1) ptx::tc_commit_multicast(&empty_bar[stage], cmask);
                        else        ptx::tc_commit(&empty_bar[stage]);
                    }
                }
            }
            sphase ^= (kPeriod / kStages) & 1;
        }
        __syncwarp();
    };
    auto run_epilogue = [&]() {
        // ===== epilogue: TMEM -> registers, running top-2 per query row =====
        constexpr int kCols = kTileN / C::kColSplit;      // train columns of a tile this warp scans
        const int quarter = warp & 3;                     // TMEM lanes [32*quarter, +32) belong to this warp
        const int mblk = (warp >> 2) & 1;                 // which 128-row query block of the CTA
        const int half = warp >> 3;                       // which column range of every tile (0 when kColSplit == 1)
        const int row_in_cta = mblk * kRowBlock + quarter * 32 + lane;
        const long long row = (long long)qb * kBlockM + row_in_cta;
        Top2<Acc> s;
        s.v1 = s.v2 = C::lowest();
        s.i1 = s.i2 = 0;
#pragma unroll
        for (int e = 0; e < 4; ++e) s.sa[e] = s.sb[e] = 0;
        s.f = C::floor_from(0);                           // below every possible dot
        unsigned floor_code = 0;                          // largest threshold code read or published so far
        const long long first_row = kRuns ? 0ll : (long long)tile_begin * kTileN;
        const unsigned limit = (unsigned)min((long long)my_tiles * kTileN, P.nt - first_row);
        RunCursor cur;
        if constexpr (kRuns) cur.seek(R.runs, R.n_runs, tile_begin);
        // barrier addresses of the tile loop, derived from an opaque copy of the shared-memory base
        const uint32_t bars_addr = ptx::lds_volatile_u32(ptx::smem_u32(smem_base_slot)) + kABytes + kStages * kBStageBytes;
        const uint32_t unit_full_addr = bars_addr + (2 * kStages + 1) * 8;
        const uint32_t unit_empty_addr = unit_full_addr + kUnits * 8;
        int unit = mblk;                                  // (2 * i + mblk) % kUnits
        uint32_t unit_use = 0;                            // (2 * i + mblk) / kUnits
        // Shared row thresholds (kFloor): called between the issue of a tile's TMEM load and its wait.  A refresh folds in
        // the value loaded by the PREVIOUS refresh (`floor_pending`: nothing waits on the load that is issued now --
        // consuming it at once stalled the warp for an L2 round trip, ~700 cycles, in front of the release of its
        // accumulator unit; that stall, not the thresholds, was why frequent refreshes used to cost more than they
        // saved), publishes this thread's second best when it improved (a fire-and-forget atomicMax) and issues the
        // next load.  Every tile while thresholds still move fast (the first 32 tiles), every 16th later (measured sweep in
        // DESIGN.md: each refresh still costs ~50 cycles of tile time).
        unsigned floor_pending = 0;
        auto refresh_floor = [&](int i) {
            if constexpr (kFloor) {
                if (i < kFloorDenseTiles || (i & kFloorLateMask) == 0) {
                    floor_code = max(floor_code, floor_pending);
                    s.f = C::max2(s.f, C::floor_from(floor_code));
                    if (row < P.nq) {              // (the threshold kernels never run with a device-side row count)
                        unsigned* floor_ptr = P.row_floor + ((long long)b * P.nq + row);
                        const unsigned e = C::valid(s.v2) ? C::encode(s.v2) : 0u;
                        if (e > floor_code) { atomicMax(floor_ptr, e); floor_code = e; }
                        floor_pending = __ldcg(floor_ptr);
                    }
                }
            }
        };
        auto process_tile = [&](int i) {
            bounded_wait_addr(unit_full_addr + unit * 8, unit_use & 1, P.error_flag);
            ptx::tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + unit * kTileN + half * kCols;
            unsigned colbase = (unsigned)i * kTileN + half * kCols;
            bool run_edge = false;
            if constexpr (kRuns) {
                colbase = (unsigned)cur.tile * kTileN + half * kCols;
                // one uniform compare per tile; only a run's partial first and last tiles take the masking branch
                run_edge = colbase < cur.lo || colbase + kCols > cur.hi;
            }
            if constexpr (C::kColSplit == 1) {
                // all four 32-column loads are issued before the first scan so their latencies overlap
                uint32_t r0[32], r1[32], r2[32], r3[32];
                ptx::tmem_ld_32x32(taddr, r0);
                ptx::tmem_ld_32x32(taddr + 32, r1);
                ptx::tmem_ld_32x32(taddr + 64, r2);
                ptx::tmem_ld_32x32(taddr + 96, r3);
                refresh_floor(i);
                tmem_ld_fence4(r0, r1, r2, r3);
                // the accumulator unit is in registers: release it before the scan
                ptx::tc_fence_before();
                __syncwarp();
                if (ptx::elect_one()) ptx::mbar_arrive_addr(unit_empty_addr + unit * 8);
                if constexpr (kRuns) {
                    if (run_edge) {
                        mask_outside<C, 32>(r0, colbase, cur.lo, cur.hi);
                        mask_outside<C, 32>(r1, colbase + 32, cur.lo, cur.hi);
                        mask_outside<C, 32>(r2, colbase + 64, cur.lo, cur.hi);
                        mask_outside<C, 32>(r3, colbase + 96, cur.lo, cur.hi);
                    }
                } else if (colbase + kCols > limit) {     // last tile of the train set only
                    mask_tail<C, 32>(r0, colbase, limit);
                    mask_tail<C, 32>(r1, colbase + 32, limit);
                    mask_tail<C, 32>(r2, colbase + 64, limit);
                    mask_tail<C, 32>(r3, colbase + 96, limit);
                }
                scan_chunk<C, kMode>(r0, colbase, s);
                scan_chunk<C, kMode>(r1, colbase + 32, s);
                scan_chunk<C, kMode>(r2, colbase + 64, s);
                scan_chunk<C, kMode>(r3, colbase + 96, s);
            } else {
                static_assert(kCols == 64, "column split");
                uint32_t r[64];
                ptx::tmem_ld_32x64(taddr, r);
                refresh_floor(i);
                tmem_ld_fence64(r);
                ptx::tc_fence_before();
                __syncwarp();
                if (ptx::elect_one()) ptx::mbar_arrive_addr(unit_empty_addr + unit * 8);
                // (tried and slower, C4 cycles per tile against 785: warp-uniform votes around the insertion path 871;
                // software pipelining over half items -- two 32-register buffers, the next item's first half loaded
                // while this item's second half is scanned -- 882.  The flat 64-column tree below measured 867 then;
                // with the group-level scan it measured a wash and was adopted, DESIGN.md §3.3 items 10-11.)
                if constexpr (kRuns) {
                    if (run_edge) mask_outside<C, 64>(r, colbase, cur.lo, cur.hi);
                } else {
                    mask_tail<C, 64>(r, colbase, limit);
                }
                scan_chunk<C, kMode, 8>(r, colbase, s);          // one compare + branch per 64 columns
            }
            unit += 2;
            if (unit >= kUnits) { unit -= kUnits; ++unit_use; }
            if constexpr (kRuns) {
                if (i + 1 < my_tiles) cur.next(R.runs);
            }
        };
#pragma unroll 1
        for (int i = 0; i < my_tiles; ++i) process_tile(i);
        const unsigned long long gbase = P.train_base + (unsigned long long)first_row;
        // exact top-2 from the saved dots of the two best groups (u64 min over (distance, trainIdx) keys = cv2's order)
        auto fold_group = [&](Acc v, unsigned i0, const uint32_t (&p)[4]) {
            if (!C::valid(v)) return;
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const Acc x = C::unpack(p[e >> 1], e & 1);
                if (C::valid(x)) top2_insert(my_keys.x, my_keys.y, ((unsigned long long)C::distance(x) << 32) | (gbase + i0 + e));
            }
        };
        fold_group(s.v1, s.i1, s.sa);
        if (kMode != 2) fold_group(s.v2, s.i2, s.sb);
        else my_keys.y = kNoMatch;
        if (half == 1) handover[row_in_cta] = my_keys;    // merged by the warp of the lower column half below
        else my_row = row;
        my_row_in_cta = row_in_cta;
    };

    // common tail; kWorker = false for the control warps, which only take part in the barriers
    auto run_tail = [&](auto worker_tag) {
        constexpr bool kWorker = decltype(worker_tag)::value;
        ptx::tc_fence_before();
        if (cs > 1) ptx::cluster_sync();   // no CTA leaves while peers may still signal its barriers
        else __syncthreads();
        if (warp == kIssuerWarp) {
            ptx::tc_fence_after();
            ptx::tmem_dealloc(tmem_base, kTmemCols);
        }
        if (kWorker && my_row >= 0 && my_row < rows_present()) {
            if constexpr (C::kColSplit == 2) {     // fold the upper column half's candidates (u64 min = cv2's order)
                const ulonglong2 o = handover[my_row_in_cta];
                top2_insert(my_keys.x, my_keys.y, o.x);
                top2_insert(my_keys.x, my_keys.y, o.y);
            }
            unsigned long long* out = P.out + (long long)split * P.out_split_stride + ((long long)b * P.nq + my_row) * 2;
            *reinterpret_cast<ulonglong2*>(out) = my_keys;
            if (!P.counters) select_candidate(P.sel, b, my_keys);      // unsplit launch: these are the row's final keys
        }
        // ---- in-kernel merge of the train splits: the last CTA of this query block folds all partials ----
        if (P.counters) {
            int* flag = reinterpret_cast<int*>(tmem_base_slot + 1);
            if (last_cta_arrives(&P.counters[(long long)b * gridDim.x + qb], (unsigned)P.splits, flag)) {
                const long long row = (long long)qb * kBlockM + threadIdx.x;
                const bool has_row = kWorker && threadIdx.x < kBlockM && row < rows_present();
                ulonglong2 k = make_ulonglong2(kNoMatch, kNoMatch);
                if (has_row) fold_partials(P.out, P.splits, P.out_split_stride, (long long)b * P.nq + row, k.x, k.y);
                // sharded database: push to the peer GPUs, wait for theirs, merge -- still inside this launch
                // (only query blocks that hold rows take part: hm_exchange_merge_kernel on a peer covers exactly
                // ceil(nq / 256) blocks, so both kernels post and wait on the same flags whatever mix of them the ranks run)
                if (P.xch.world > 1 && (long long)qb * kBlockM < P.nq) k = exchange_and_merge(P.xch, row, has_row, k, qb);
                if (has_row) {
                    *reinterpret_cast<ulonglong2*>(P.final_out + ((long long)b * P.nq + row) * 2) = k;
                    select_candidate(P.sel, b, k);
                }
            }
        }
        if (kWorker && threadIdx.x == 0 && (blockIdx.x | blockIdx.y | blockIdx.z) == 0 && P.clock_probe) {
            unsigned long long t;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            P.clock_probe[2] = (long long)t;
            P.clock_probe[3] = clock64();
        }
    };

    if constexpr (C::kRegisterHandover) {
        // Register handover: the control warpgroup (producer, issuer, two idle warps) drops to 32 registers and never
        // comes back -- its whole remaining path, tail included, is compiled under that budget -- and the epilogue
        // warps rise to 112 (4 x 32 + 16 x 112 = 20 x 96, the registers the CTA was launched with).
        if (warp >= kProducerWarp) {
            asm volatile("setmaxnreg.dec.sync.aligned.u32 32;\n");
            if (warp == kProducerWarp) run_producer();
            else if (warp == kIssuerWarp) run_issuer();
            run_tail(std::false_type{});
            return;
        }
        asm volatile("setmaxnreg.inc.sync.aligned.u32 112;\n");
        run_epilogue();
        run_tail(std::true_type{});
    } else {
        if (warp == kProducerWarp) run_producer();
        else if (warp == kIssuerWarp) run_issuer();
        else run_epilogue();
        run_tail(std::true_type{});
    }
}

__global__ void __launch_bounds__(threads<CoreI8>(), 1) hm_i8_knn2_kernel(const TcParams P) { tc_knn2_body<CoreI8, 0>(P); }
__global__ void __launch_bounds__(threads<CoreF4>(), 1) hm_f4_knn2_kernel(const TcParams P) { tc_knn2_body<CoreF4, 0>(P); }
// the same kernels with the shared row thresholds (TcParams::row_floor): launched when the train set is split
// over many short CTAs per query row
__global__ void __launch_bounds__(threads<CoreI8>(), 1) hm_i8_knn2_floor_kernel(const TcParams P) { tc_knn2_body<CoreI8, 1>(P); }
__global__ void __launch_bounds__(threads<CoreF4>(), 1) hm_f4_knn2_floor_kernel(const TcParams P) { tc_knn2_body<CoreF4, 1>(P); }
// nearest neighbour only (second key = HM_NO_MATCH): the swapped pass of the mutual check
__global__ void __launch_bounds__(threads<CoreI8>(), 1) hm_i8_knn1_kernel(const TcParams P) { tc_knn2_body<CoreI8, 2>(P); }
__global__ void __launch_bounds__(threads<CoreF4>(), 1) hm_f4_knn1_kernel(const TcParams P) { tc_knn2_body<CoreF4, 2>(P); }

// top-2 over the selected runs of a resident shard (hm_knn2_resident_runs*): the same bodies walking RunArgs; the floor
// kernels for split launches, the plain ones for unsplit shapes, the fused exchange through TcParams::xch as above
__global__ void __launch_bounds__(threads<CoreI8>(), 1) hm_i8_knn2_runs_kernel(const TcParams P, const RunArgs R) { tc_knn2_body<CoreI8, 0, true>(P, R); }
__global__ void __launch_bounds__(threads<CoreF4>(), 1) hm_f4_knn2_runs_kernel(const TcParams P, const RunArgs R) { tc_knn2_body<CoreF4, 0, true>(P, R); }
__global__ void __launch_bounds__(threads<CoreI8>(), 1) hm_i8_knn2_runs_floor_kernel(const TcParams P, const RunArgs R) { tc_knn2_body<CoreI8, 1, true>(P, R); }
__global__ void __launch_bounds__(threads<CoreF4>(), 1) hm_f4_knn2_runs_floor_kernel(const TcParams P, const RunArgs R) { tc_knn2_body<CoreF4, 1, true>(P, R); }

using KernelFn = void (*)(const TcParams);
template <class C> KernelFn kernel_of(int mode = 0);
template <> KernelFn kernel_of<CoreI8>(int mode) { return mode == 1 ? hm_i8_knn2_floor_kernel : mode == 2 ? hm_i8_knn1_kernel : hm_i8_knn2_kernel; }
template <> KernelFn kernel_of<CoreF4>(int mode) { return mode == 1 ? hm_f4_knn2_floor_kernel : mode == 2 ? hm_f4_knn1_kernel : hm_f4_knn2_kernel; }
using RunsKernelFn = void (*)(const TcParams, const RunArgs);
template <class C> RunsKernelFn runs_kernel_of(bool floor);
template <> RunsKernelFn runs_kernel_of<CoreI8>(bool floor) { return floor ? hm_i8_knn2_runs_floor_kernel : hm_i8_knn2_runs_kernel; }
template <> RunsKernelFn runs_kernel_of<CoreF4>(bool floor) { return floor ? hm_f4_knn2_runs_floor_kernel : hm_f4_knn2_runs_kernel; }

struct TcPlan {
    int ntiles, splits, tiles_per_split;
    int cluster;                     // CTAs per cluster (query blocks sharing the B tiles)
    long long qblocks;               // grid.x, rounded up to a multiple of `cluster`
};

// test hook: HM_I8_CLUSTER=1|2|4 forces the cluster size of every tensor-core launch of the process, so that tests can
// run cluster shapes the planner would not choose for their problem size
int cluster_override()
{
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("HM_I8_CLUSTER");
        v = e ? atoi(e) : 0;
        if (v != 1 && v != 2 && v != 4) v = 0;
    }
    return v;
}

// Per-device launch state.  cudaFuncSetAttribute (the > 48 KB dynamic shared memory opt-in) and cluster occupancy
// are per DEVICE, and one process may drive several devices (BFMatcher(device=...), FrameDescriptorStore(device=...)),
// from several threads: both caches are keyed by the device ordinal and guarded by one mutex.
constexpr int kMaxDevices = 64;
std::mutex g_launch_state_mu;

int current_device_slot()
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); dev = 0; }
    return (dev >= 0 && dev < kMaxDevices) ? dev : -1;      // -1: do not cache
}

template <class C>
cudaError_t ensure_smem_opt_in()
{
    static bool done[kMaxDevices] = {};
    const int dev = current_device_slot();
    std::lock_guard<std::mutex> lock(g_launch_state_mu);
    if (dev >= 0 && done[dev]) return cudaSuccess;
    for (int mode = 0; mode < 3; ++mode) {
        const cudaError_t e = cudaFuncSetAttribute(kernel_of<C>(mode), cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes<C>());
        if (e != cudaSuccess) return e;
    }
    for (int floor = 0; floor < 2; ++floor) {
        const cudaError_t e = cudaFuncSetAttribute(runs_kernel_of<C>(floor != 0), cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes<C>());
        if (e != cudaSuccess) return e;
    }
    if (dev >= 0) done[dev] = true;
    return cudaSuccess;
}

// CTAs that can be co-resident when launched as clusters of `cs` (1 CTA per SM; clusters of 4 cannot
// use every SM of every GPC).  Queried once per device and cluster size; falls back to the SM count.
template <class C>
int resident_ctas(int cs, int sm_count)
{
    static int cache[kMaxDevices][5] = {};
    if (cs <= 1) return sm_count;
    const int dev = current_device_slot();
    if (dev >= 0) {
        std::lock_guard<std::mutex> lock(g_launch_state_mu);
        if (cache[dev][cs]) return cache[dev][cs];
    }
    int v = sm_count;
    if (ensure_smem_opt_in<C>() == cudaSuccess) {
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3(cs * 64, 1, 1);
        cfg.blockDim = dim3(threads<C>());
        cfg.dynamicSmemBytes = smem_bytes<C>();
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = (unsigned)cs;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        int n = 0;
        if (cudaOccupancyMaxActiveClusters(&n, kernel_of<C>(), &cfg) == cudaSuccess && n > 0) v = n * cs;
        else cudaGetLastError();
    } else {
        cudaGetLastError();
    }
    if (dev >= 0) {
        std::lock_guard<std::mutex> lock(g_launch_state_mu);
        cache[dev][cs] = v;
    }
    return v;
}

template <class C>
TcPlan plan_tc_cluster(long long nq, long long nt, int batch, int sm_count, int cluster)
{
    TcPlan pl{};
    const long long qb = ceil_div(nq, kBlockM);
    pl.cluster = cluster;
    pl.qblocks = ceil_div(qb, pl.cluster) * pl.cluster;
    sm_count = resident_ctas<C>(pl.cluster, sm_count);
    pl.ntiles = (int)ceil_div(nt, C::kTileN);
    const long long items = pl.qblocks * batch;
    // choose the split count minimising (waves) x (tiles per CTA + fixed prologue worth a few tiles)
    long long best_cost = -1;
    int best = 1;
    const int max_splits = (int)min((long long)pl.ntiles, 4096ll);
    for (int s = 1; s <= max_splits; ++s) {
        const long long tps = ceil_div(pl.ntiles, s);
        const long long real_s = ceil_div(pl.ntiles, tps);
        const long long waves = ceil_div(items * real_s, sm_count);
        const long long cost = waves * (tps + C::kPrologueTiles);
        if (best_cost < 0 || cost < best_cost) {
            best_cost = cost;
            best = s;
        }
        if (items * s > 16ll * sm_count) break;
    }
    pl.tiles_per_split = (int)ceil_div(pl.ntiles, best);
    pl.splits = (int)ceil_div(pl.ntiles, pl.tiles_per_split);
    return pl;
}

template <class C>
TcPlan plan_tc(long long nq, long long nt, int batch, int sm_count)
{
    if (cluster_override()) return plan_tc_cluster<C>(nq, nt, batch, sm_count, cluster_override());
    // Pairs of query blocks share every train tile through multicast: half the L2 reads, 1.7 % on C4 (690 vs 702 cycles
    // per tile at 1730 tiles per CTA; clusters of 4 lose SMs to GPC packing: 747).  CTAs that see few tiles gain nothing
    // from it and schedule better alone: C5 (79 tiles per CTA) +2 %, C2 (16) +2.5 %, 16k x 16k +2.5 %, and a wash for
    // the 2000-query shards of the multi-GPU runs (445-889 tiles: within 0.7 %).  Clusters of 2 therefore pay from this
    // many tiles per CTA on:
    constexpr int kClusterMinTiles = 1024;
    if (ceil_div(nq, kBlockM) >= 2) {
        const TcPlan pl = plan_tc_cluster<C>(nq, nt, batch, sm_count, 2);
        if (pl.tiles_per_split >= kClusterMinTiles) return pl;
    }
    return plan_tc_cluster<C>(nq, nt, batch, sm_count, 1);
}

// rows of a prepared image: whole tiles of the core's height, rounded up to whole 256-row query blocks
template <class C>
long long padded_rows(long long n) { return ceil_div(ceil_div(n, C::kTileN) * C::kTileN, kPadRows) * kPadRows; }

// workspace layout: [256 B][arrival counters | shared row thresholds][partials][prepared q][prepared t]
template <class C>
size_t partials_bytes(long long nq, long long nt, int batch, int sm_count)
{
    const TcPlan pl = plan_tc<C>(nq, nt, batch, sm_count);
    return (size_t)pl.splits * batch * nq * 2 * sizeof(unsigned long long);   // also when splits == 1 (partials mode)
}

// arrival counters followed by one 32-bit threshold code per query row (one memset clears both)
inline size_t zeroed_bytes(long long row_blocks, long long rows) { return counters_bytes(row_blocks) + counters_bytes((rows + 1) / 2 * 2); }

template <class C>
size_t workspace_bytes_of(long long nq, long long nt, int batch, int sm_count, bool with_prepare)
{
    size_t b = 256 + zeroed_bytes(plan_tc<C>(nq, nt, batch, sm_count).qblocks * batch, nq * batch) + partials_bytes<C>(nq, nt, batch, sm_count);
    b = (b + 1023) & ~(size_t)1023;
    if (with_prepare) b += (size_t)(padded_rows<C>(nq) + padded_rows<C>(nt)) * C::kRowBytes * batch;
    return b;
}

template <class C>
int launch_prepared(const void* qprep, long long nq, const void* tprep, long long nt, int batch,
                    unsigned long long train_base, unsigned long long* out, void* ws, size_t ws_bytes,
                    int sm_count, cudaStream_t stream, const unsigned long long** out_partials,
                    int* out_groups, const ExchangeArgs* exchange, bool top1 = false, const QueryBits* qbits = nullptr,
                    const SelectArgs* select = nullptr, const RunArgs* runs = nullptr, long long run_tiles = 0)
{
    HM_CUDA_CHECK(ensure_smem_opt_in<C>());
    // a run walk is planned over its virtual tiles exactly as a whole train set over its tiles
    const long long plan_nt = runs ? run_tiles * C::kTileN : nt;
    const TcPlan pl = plan_tc<C>(nq, plan_nt, batch, sm_count);
    if (ceil_div(nt, C::kTileN) * C::kTileN > (1ll << 32)) {
        set_error("train set too large for 32-bit trainIdx");
        return HM_ERR_UNSUPPORTED;
    }
    if (runs && (batch != 1 || top1 || (qbits && qbits->index) || (select && select->slot_of) || out == nullptr)) {
        set_error("a run walk is a single top-2 problem with an output buffer");
        return HM_ERR_INVALID_ARGUMENT;
    }
    const bool keep_partials = out == nullptr;
    const size_t cbytes = zeroed_bytes(pl.qblocks * batch, nq * batch);
    const size_t need = 256 + cbytes + partials_bytes<C>(nq, plan_nt, batch, sm_count);
    if (!ws || ws_bytes < need) {
        set_error("workspace too small: need %zu bytes, got %zu", need, ws_bytes);
        return HM_ERR_WORKSPACE;
    }
    TcParams P{};
    if (qbits && qbits->bits) {
        if (!C::kScales) {
            set_error("in-kernel query expansion exists for the kind::mxf4 core only");
            return HM_ERR_UNSUPPORTED;
        }
        P.qbits = qbits->bits; P.q_bits_stride = qbits->stride; P.q_bits_batch_stride = qbits->batch_stride;
        P.q_index = qbits->index; P.q_index_batch_stride = qbits->index_batch_stride; P.nq_dyn = qbits->nq_dyn;
    }
    if (select && select->slot_of) {
        if (keep_partials || (exchange && exchange->world > 1)) {
            set_error("candidate selection needs final keys of a single GPU");
            return HM_ERR_INVALID_ARGUMENT;
        }
        P.sel = *select;
    }
    P.qprep = static_cast<const uint8_t*>(qprep);
    P.tprep = static_cast<const uint8_t*>(tprep);
    P.nq = nq; P.nt = nt;
    P.q_padded = padded_rows<C>(nq);
    P.t_padded = padded_rows<C>(nt);
    P.tiles_per_split = pl.tiles_per_split;
    P.ntiles = pl.ntiles;            // run walk: the virtual tiles
    P.train_base = train_base;
    P.error_flag = static_cast<int*>(ws);
    P.clock_probe = reinterpret_cast<long long*>(static_cast<uint8_t*>(ws) + HM_WS_CLOCK_PROBE_OFFSET);   // inside the 256-byte header
    P.q_blocks_valid = P.q_padded / kBlockM;
    const long long rows = nq * batch;
    unsigned* counters = reinterpret_cast<unsigned*>(static_cast<uint8_t*>(ws) + 256);
    unsigned long long* partials = reinterpret_cast<unsigned long long*>(static_cast<uint8_t*>(ws) + 256 + cbytes);
    P.splits = pl.splits;
    if (pl.splits > 1 || keep_partials) {
        P.out = partials;
        P.out_split_stride = rows * 2;
    }
    const bool fused_exchange = exchange && exchange->world > 1;
    if (fused_exchange) {
        if (batch != 1 || keep_partials) {
            set_error("fused exchange needs batch == 1 and an output buffer");
            return HM_ERR_INVALID_ARGUMENT;
        }
        static_assert(kBlockM == kExchangeRows, "flag granularity = query block");
        P.xch = *exchange;
        P.out = partials;                  // even with one split: the exchange runs in the last-CTA path
        P.out_split_stride = rows * 2;
    }
    // shared row thresholds: between the CTAs of a query row in split launches (and, with kColSplit == 2, between the
    // two column-half warps of the row in each CTA)
    bool zero_block = false;
    const bool floor_eligible = !top1 && !P.nq_dyn && pl.splits > 1;
    if (floor_eligible) {
        P.row_floor = reinterpret_cast<unsigned*>(reinterpret_cast<uint8_t*>(counters) + counters_bytes(pl.qblocks * batch));
        zero_block = true;
    }
    if ((pl.splits > 1 || fused_exchange) && !keep_partials) {   // merge in-kernel: last CTA per query block writes `out`
        P.counters = counters;
        P.final_out = out;
        zero_block = true;
    } else if (!(pl.splits > 1 || keep_partials)) {
        P.out = out;
        P.out_split_stride = 0;
    }
    if (zero_block) HM_CUDA_CHECK(cudaMemsetAsync(counters, 0, cbytes, stream));
    if (pl.qblocks > 0x7FFFFFFFll || pl.splits > 65535 || batch > 65535) {
        set_error("grid too large");
        return HM_ERR_UNSUPPORTED;
    }
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)pl.qblocks, (unsigned)pl.splits, (unsigned)batch);
    cfg.blockDim = dim3(threads<C>());
    cfg.dynamicSmemBytes = smem_bytes<C>();
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)pl.cluster;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    profile_mark(true, stream);
    cudaError_t le = runs ? cudaLaunchKernelEx(&cfg, runs_kernel_of<C>(P.row_floor != nullptr), P, *runs)
                          : cudaLaunchKernelEx(&cfg, kernel_of<C>(P.row_floor ? 1 : top1 ? 2 : 0), P);
    profile_mark(false, stream);
    if (le != cudaSuccess) {
        set_error("cudaLaunchKernelEx(tensor-core k-NN kernel, cluster %d) failed: %s", pl.cluster, cudaGetErrorString(le));
        return HM_ERR_CUDA;
    }
    HM_CUDA_CHECK(cudaGetLastError());
    if (keep_partials) {
        if (out_partials) *out_partials = partials;
        if (out_groups) *out_groups = pl.splits;
    }
    return HM_OK;
}

template <class C>
int launch_prepare_of(const uint8_t* bits, long long n, long long stride, long long batch_stride, int batch,
                      void* prepared, cudaStream_t stream)
{
    if (n <= 0 || batch <= 0) return HM_OK;
    PrepareParams P{};
    P.bits = bits; P.n = n; P.stride = stride; P.batch_stride = batch_stride;
    P.padded_rows = padded_rows<C>(n);
    P.out = static_cast<uint8_t*>(prepared);
    const long long chunks = P.padded_rows * (C::kRowBytes / 16);
    dim3 grid((unsigned)ceil_div(chunks, 256), (unsigned)batch);
    if (C::kScales) hm_prepare_f4_kernel<<<grid, 256, 0, stream>>>(P);
    else            hm_prepare_kernel<<<grid, 256, 0, stream>>>(P);
    HM_CUDA_CHECK(cudaGetLastError());
    return HM_OK;
}

template <class C>
int launch_knn2_of(const KnnProblem& p, unsigned long long* out, void* ws, size_t ws_bytes, int sm_count, cudaStream_t stream)
{
    const size_t need = workspace_bytes_of<C>(p.nq, p.nt, p.batch, sm_count, true);
    if (!ws || ws_bytes < need) {
        set_error("workspace too small: need %zu bytes, got %zu", need, ws_bytes);
        return HM_ERR_WORKSPACE;
    }
    const size_t head = workspace_bytes_of<C>(p.nq, p.nt, p.batch, sm_count, false);
    uint8_t* qprep = static_cast<uint8_t*>(ws) + head;
    uint8_t* tprep = qprep + (size_t)padded_rows<C>(p.nq) * C::kRowBytes * p.batch;
    int rc = HM_OK;
    QueryBits qb{};
    if (C::kScales) {           // kind::mxf4: the k-NN kernel expands the query rows itself
        qb.bits = p.q; qb.stride = p.q_stride; qb.batch_stride = p.q_batch_stride;
    } else {
        rc = launch_prepare_of<C>(p.q, p.nq, p.q_stride, p.q_batch_stride, p.batch, qprep, stream);
        if (rc != HM_OK) return rc;
    }
    rc = launch_prepare_of<C>(p.t, p.nt, p.t_stride, p.t_batch_stride, p.batch, tprep, stream);
    if (rc != HM_OK) return rc;
    if (p.select && !C::kScales) {
        set_error("candidate selection exists for the kind::mxf4 core only");
        return HM_ERR_UNSUPPORTED;
    }
    return launch_prepared<C>(qprep, p.nq, tprep, p.nt, p.batch, p.train_base, out, ws, head, sm_count, stream, nullptr,
                              nullptr, nullptr, p.top1, &qb, p.select);
}

}  // namespace

// ---- core dispatch (variant must be HM_VARIANT_I8 or HM_VARIANT_F4) ---------------------------
size_t prepared_bytes(long long n, int variant)
{
    return variant == HM_VARIANT_F4 ? (size_t)padded_rows<CoreF4>(n) * CoreF4::kRowBytes : (size_t)padded_rows<CoreI8>(n) * CoreI8::kRowBytes;
}

int launch_prepare(const uint8_t* bits, long long n, long long stride, long long batch_stride, int batch,
                   void* prepared, int variant, cudaStream_t stream)
{
    return variant == HM_VARIANT_F4 ? launch_prepare_of<CoreF4>(bits, n, stride, batch_stride, batch, prepared, stream)
                                    : launch_prepare_of<CoreI8>(bits, n, stride, batch_stride, batch, prepared, stream);
}

size_t tc_workspace_bytes(long long nq, long long nt, int batch, int sm_count, bool with_prepare, int variant)
{
    return variant == HM_VARIANT_F4 ? workspace_bytes_of<CoreF4>(nq, nt, batch, sm_count, with_prepare)
                                    : workspace_bytes_of<CoreI8>(nq, nt, batch, sm_count, with_prepare);
}

int launch_tc_knn2_prepared(const void* qprep, long long nq, const void* tprep, long long nt, int batch,
                            unsigned long long train_base, unsigned long long* out, void* ws, size_t ws_bytes,
                            int sm_count, int variant, cudaStream_t stream, const unsigned long long** out_partials,
                            int* out_groups, const ExchangeArgs* exchange)
{
    return variant == HM_VARIANT_F4
               ? launch_prepared<CoreF4>(qprep, nq, tprep, nt, batch, train_base, out, ws, ws_bytes, sm_count, stream,
                                         out_partials, out_groups, exchange)
               : launch_prepared<CoreI8>(qprep, nq, tprep, nt, batch, train_base, out, ws, ws_bytes, sm_count, stream,
                                         out_partials, out_groups, exchange);
}

// resident database, query as packed bits: kind::mxf4 expands the query inside the k-NN kernel; kind::i8 expands it into
// the tail of the workspace first (ws_bytes must be tc_resident_workspace_bytes)
size_t tc_resident_workspace_bytes(long long nq, long long nt, int sm_count, int variant)
{
    size_t b = (tc_workspace_bytes(nq, nt, 1, sm_count, false, variant) + 1023) & ~(size_t)1023;
    if (variant != HM_VARIANT_F4) b += prepared_bytes(nq, variant);
    return b;
}

// runs != nullptr: the walk over the selected runs, planned and sized over run_tiles tiles instead of nt rows
static int resident_of(const uint8_t* qbits, long long nq, long long q_stride, const void* tprep, long long nt,
                       unsigned long long train_base, unsigned long long* out, void* ws, size_t ws_bytes, int sm_count,
                       int variant, cudaStream_t stream, const ExchangeArgs* exchange, const RunArgs* runs,
                       long long run_tiles)
{
    const long long plan_nt = runs ? run_tiles * kRowBlock : nt;
    const size_t need = tc_resident_workspace_bytes(nq, plan_nt, sm_count, variant);
    if (!ws || ws_bytes < need) {
        set_error("workspace too small: need %zu bytes, got %zu", need, ws_bytes);
        return HM_ERR_WORKSPACE;
    }
    if (variant == HM_VARIANT_F4) {
        QueryBits qb{qbits, q_stride, 0};
        return launch_prepared<CoreF4>(nullptr, nq, tprep, nt, 1, train_base, out, ws, ws_bytes, sm_count, stream, nullptr,
                                       nullptr, exchange, false, &qb, nullptr, runs, run_tiles);
    }
    const size_t head = (tc_workspace_bytes(nq, plan_nt, 1, sm_count, false, variant) + 1023) & ~(size_t)1023;
    uint8_t* qprep = static_cast<uint8_t*>(ws) + head;
    const int rc = launch_prepare_of<CoreI8>(qbits, nq, q_stride, 0, 1, qprep, stream);
    if (rc != HM_OK) return rc;
    return launch_prepared<CoreI8>(qprep, nq, tprep, nt, 1, train_base, out, ws, head, sm_count, stream, nullptr, nullptr,
                                   exchange, false, nullptr, nullptr, runs, run_tiles);
}

int launch_tc_knn2_resident(const uint8_t* qbits, long long nq, long long q_stride, const void* tprep, long long nt,
                            unsigned long long train_base, unsigned long long* out, void* ws, size_t ws_bytes,
                            int sm_count, int variant, cudaStream_t stream, const ExchangeArgs* exchange)
{
    return resident_of(qbits, nq, q_stride, tprep, nt, train_base, out, ws, ws_bytes, sm_count, variant, stream, exchange,
                       nullptr, 0);
}

int launch_tc_knn2_resident_runs(const uint8_t* qbits, long long nq, long long q_stride, const void* tprep, long long nt,
                                 const RunArgs& runs, const RunTotals& totals, unsigned long long train_base,
                                 unsigned long long* out, void* ws, size_t ws_bytes, int sm_count, int variant,
                                 cudaStream_t stream, const ExchangeArgs* exchange)
{
    return resident_of(qbits, nq, q_stride, tprep, nt, train_base, out, ws, ws_bytes, sm_count, variant, stream, exchange,
                       &runs, totals.tiles);
}

int launch_tc_knn1_candidates(const KnnProblem& p, const int* list, const int* count, unsigned long long* out, void* ws,
                              size_t ws_bytes, int sm_count, cudaStream_t stream)
{
    using C = CoreF4;
    const size_t need = workspace_bytes_of<C>(p.nq, p.nt, p.batch, sm_count, true);
    if (!ws || ws_bytes < need) {
        set_error("workspace too small: need %zu bytes, got %zu", need, ws_bytes);
        return HM_ERR_WORKSPACE;
    }
    const size_t head = workspace_bytes_of<C>(p.nq, p.nt, p.batch, sm_count, false);
    uint8_t* tprep = static_cast<uint8_t*>(ws) + head + (size_t)padded_rows<C>(p.nq) * C::kRowBytes * p.batch;
    int rc = launch_prepare_of<C>(p.t, p.nt, p.t_stride, p.t_batch_stride, p.batch, tprep, stream);
    if (rc != HM_OK) return rc;
    QueryBits qb{};
    qb.bits = p.q; qb.stride = p.q_stride; qb.batch_stride = p.q_batch_stride;
    qb.index = list; qb.index_batch_stride = p.nq; qb.nq_dyn = count;
    return launch_prepared<C>(nullptr, p.nq, tprep, p.nt, p.batch, 0, out, ws, head, sm_count, stream, nullptr, nullptr,
                              nullptr, true, &qb);
}

// "kernel grid=(x,y,z) cluster=c" of the launch the given shape would get (introspection for bench / docs)
template <class C>
static void describe_of(long long nq, long long nt, int batch, int sm_count, bool top1, char* buf, size_t n)
{
    const TcPlan pl = plan_tc<C>(nq, nt, batch, sm_count);
    const bool floor = !top1 && pl.splits > 1;
    snprintf(buf, n, "hm_%s_knn%s%s_kernel grid=(%lld,%d,%d) cluster=%d tiles_per_cta=%d", C::kScales ? "f4" : "i8",
             top1 ? "1" : "2", floor ? "_floor" : "", pl.qblocks, pl.splits, batch, pl.cluster, pl.tiles_per_split);
}

void describe_tc_launch(long long nq, long long nt, int batch, int sm_count, int variant, bool top1, char* buf, size_t n)
{
    if (variant == HM_VARIANT_F4) describe_of<CoreF4>(nq, nt, batch, sm_count, top1, buf, n);
    else                          describe_of<CoreI8>(nq, nt, batch, sm_count, top1, buf, n);
}

template <class C>
static void describe_runs_of(long long nq, const long long* runs4, int n_runs, long long tiles, int sm_count, char* buf,
                             size_t n, long long* pieces)
{
    const TcPlan pl = plan_tc<C>(nq, tiles * C::kTileN, 1, sm_count);
    if (buf && n) {
        snprintf(buf, n, "hm_%s_knn2_runs%s_kernel grid=(%lld,%d,1) cluster=%d tiles_per_cta=%d run_tiles=%lld",
                 C::kScales ? "f4" : "i8", pl.splits > 1 ? "_floor" : "", pl.qblocks, pl.splits, pl.cluster,
                 pl.tiles_per_split, tiles);
    }
    if (!pieces) return;
    for (int s = 0; s < pl.splits; ++s) {
        const long long v0 = (long long)s * pl.tiles_per_split, v1 = min(v0 + pl.tiles_per_split, tiles);
        RunCursor cur;
        cur.seek(runs4, n_runs, v0);
        for (long long v = v0; v < v1; ++v) {
            long long* p = pieces + 4 * v;
            p[0] = s;
            p[1] = cur.tile;
            p[2] = max((long long)cur.tile * kRowBlock, (long long)cur.lo);
            p[3] = min((long long)(cur.tile + 1) * kRowBlock, (long long)cur.hi);
            if (v + 1 < v1) cur.next(runs4);
        }
    }
}

void describe_tc_runs(long long nq, const long long* runs_host4, int n_runs, long long tiles, int sm_count, int variant,
                      char* buf, size_t n, long long* pieces)
{
    if (variant == HM_VARIANT_F4) describe_runs_of<CoreF4>(nq, runs_host4, n_runs, tiles, sm_count, buf, n, pieces);
    else                          describe_runs_of<CoreI8>(nq, runs_host4, n_runs, tiles, sm_count, buf, n, pieces);
}

int launch_tc_knn2(const KnnProblem& p, unsigned long long* out, void* ws, size_t ws_bytes, int sm_count, int variant,
                   cudaStream_t stream)
{
    return variant == HM_VARIANT_F4 ? launch_knn2_of<CoreF4>(p, out, ws, ws_bytes, sm_count, stream)
                                    : launch_knn2_of<CoreI8>(p, out, ws, ws_bytes, sm_count, stream);
}

}  // namespace hm
