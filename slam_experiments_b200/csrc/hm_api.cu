// C ABI of the matcher (include/hm_matcher.h): argument validation, variant selection,
// workspace carving, launch sequencing.  No CPU fallback anywhere: without an sm_100
// device every compute entry point fails with HM_ERR_NO_DEVICE.
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <new>
#include <vector>

#include "hm_common.cuh"

namespace hm {

static thread_local char g_error[512] = "";

void set_error(const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}

static thread_local cudaEvent_t g_prof_start = nullptr, g_prof_stop = nullptr;
static thread_local bool g_prof_armed = false;

// The event pair brackets the FIRST dominant-kernel launch after hm_profile_events() armed it: the forward k-NN of a
// pipeline call (its swapped / candidate pass is not the kernel the roofline line is about).
void profile_mark(bool start, cudaStream_t stream)
{
    if (!g_prof_armed || !g_prof_start || !g_prof_stop) return;
    cudaEventRecord(start ? g_prof_start : g_prof_stop, stream);
    if (!start) g_prof_armed = false;
}

int device_info(DeviceInfo* out)
{
    static std::mutex mu;
    static DeviceInfo cache[64];
    static bool have[64] = {false};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("no CUDA device: %s (this library has no CPU fallback)", cudaGetErrorString(e));
        return HM_ERR_NO_DEVICE;
    }
    std::lock_guard<std::mutex> lock(mu);
    if (dev < 0 || dev >= 64) {
        set_error("device ordinal %d out of range", dev);
        return HM_ERR_NO_DEVICE;
    }
    if (!have[dev]) {
        DeviceInfo d{};
        d.device = dev;
        if (cudaDeviceGetAttribute(&d.sm_count, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
            cudaDeviceGetAttribute(&d.cc_major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess ||
            cudaDeviceGetAttribute(&d.cc_minor, cudaDevAttrComputeCapabilityMinor, dev) != cudaSuccess) {
            cudaGetLastError();
            set_error("cudaDeviceGetAttribute failed");
            return HM_ERR_CUDA;
        }
        if (d.cc_major != 10) {
            set_error("device %d is sm_%d%d; this library is built for sm_100a only", dev, d.cc_major, d.cc_minor);
            return HM_ERR_NO_DEVICE;
        }
        cache[dev] = d;
        have[dev] = true;
    }
    *out = cache[dev];
    return HM_OK;
}

namespace {

inline size_t align_up(size_t v, size_t a = 256) { return (v + a - 1) / a * a; }

// Static per-shape table (DESIGN.md, "variant selection"): the tensor-core variant pays an
// operand-expansion pre-pass (two more launches, ~3 us each); kernel-only times (profiles/r01p_probe_shapes.txt):
// 2000 x 2000 POPC 22 us vs tensor 15 + 6 us, 4096 x 4096 52 us vs 22 + 6 us -- crossover near 8e6 pairs.
// The tensor-core core AUTO resolves to.
int default_tensor_variant() { return HM_DEFAULT_TENSOR_VARIANT; }

int select_variant(long long nq, long long nt, int batch)
{
    const double pairs = (double)nq * (double)nt * (double)batch;
    if (nq >= 64 && nt >= 256 && pairs >= 8.0e6) return default_tensor_variant();
    return HM_VARIANT_POPC;
}

int resolve_variant(int variant, long long nq, long long nt, int batch)
{
    if (variant == HM_VARIANT_AUTO) return select_variant(nq, nt, batch);
    return variant;
}

// prepared-operand entry points: AUTO = the default tensor core; POPC has no prepared form
int resolve_tensor_variant(int variant)
{
    if (variant == HM_VARIANT_AUTO) return default_tensor_variant();
    if (variant == HM_VARIANT_I8 || variant == HM_VARIANT_F4) return variant;
    set_error("variant %d has no prepared operand format (expected HM_VARIANT_I8, HM_VARIANT_F4 or AUTO)", variant);
    return HM_ERR_INVALID_ARGUMENT;
}

int check_rows(const void* p, long long n, long long stride, const char* what)
{
    if (n < 0) {
        set_error("%s: negative row count", what);
        return HM_ERR_INVALID_ARGUMENT;
    }
    if (n == 0) return HM_OK;
    if (!p) {
        set_error("%s: null pointer", what);
        return HM_ERR_INVALID_ARGUMENT;
    }
    if ((reinterpret_cast<uintptr_t>(p) & 15) || stride < HM_DESC_BYTES || (stride & 15)) {
        set_error("%s: base must be 16-byte aligned and row stride a multiple of 16 >= 32 (got stride %lld)", what,
                  stride);
        return HM_ERR_INVALID_ARGUMENT;
    }
    return HM_OK;
}

size_t knn_workspace(long long nq, long long nt, int batch, int variant, int sm_count)
{
    if (nq <= 0 || nt <= 0 || batch <= 0) return 0;
    size_t a = 0, b = 0;
    if (variant == HM_VARIANT_AUTO || variant == HM_VARIANT_POPC) a = popc_workspace_bytes(nq, nt, batch, sm_count);
    if (variant == HM_VARIANT_AUTO) variant = default_tensor_variant();
    if (variant == HM_VARIANT_I8 || variant == HM_VARIANT_F4) b = tc_workspace_bytes(nq, nt, batch, sm_count, true, variant);
    return align_up(a > b ? a : b);
}

// candidate selection of the mutual check: [count: batch ints, padded | slot_of: batch x nt ints] (zeroed per call)
// followed by [list: batch x nt ints]
inline size_t select_zeroed_bytes(long long nt, int batch) { return align_up((size_t)batch * 4) + align_up((size_t)batch * nt * 4); }
inline size_t select_bytes(long long nt, int batch) { return select_zeroed_bytes(nt, batch) + align_up((size_t)batch * nt * 4); }

__global__ void hm_fill_keys_kernel(unsigned long long* p, long long n)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = kNoMatch;
}

int fill_no_match(unsigned long long* out, long long n, cudaStream_t stream)
{
    if (n <= 0) return HM_OK;
    hm_fill_keys_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, stream>>>(out, n);
    HM_CUDA_CHECK(cudaGetLastError());
    return HM_OK;
}

int knn2_dispatch(const KnnProblem& p, unsigned long long* out, int variant, void* ws, size_t ws_bytes,
                  cudaStream_t stream)
{
    DeviceInfo di;
    int rc = device_info(&di);
    if (rc != HM_OK) return rc;
    if (p.batch <= 0 || p.nq == 0) return HM_OK;
    if (!out) {
        set_error("out_keys is null");
        return HM_ERR_INVALID_ARGUMENT;
    }
    if ((rc = check_rows(p.q, p.nq, p.q_stride, "query")) != HM_OK) return rc;
    if ((rc = check_rows(p.t, p.nt, p.t_stride, "train")) != HM_OK) return rc;
    if (p.nt == 0) return fill_no_match(out, p.nq * p.batch * 2, stream);   // knnMatch: Nq empty rows (SURVEY E3)
    if (p.batch > 1 && ((p.q_batch_stride & 15) || (p.t_batch_stride & 15))) {
        set_error("batch strides must be multiples of 16 bytes");
        return HM_ERR_INVALID_ARGUMENT;
    }
    const int v = resolve_variant(variant, p.nq, p.nt, p.batch);
    switch (v) {
        case HM_VARIANT_POPC: return launch_popc_knn2(p, out, ws, ws_bytes, di.sm_count, stream);
        case HM_VARIANT_I8:
        case HM_VARIANT_F4: return launch_tc_knn2(p, out, ws, ws_bytes, di.sm_count, v, stream);
        default: set_error("unknown variant %d", variant); return HM_ERR_INVALID_ARGUMENT;
    }
}


// ---- selections of train rows as runs (hm_knn2_resident_runs, hm_knn2_runs) ----------------------------------------
// runs_host[n_runs][2] must be non-empty, ascending and disjoint within [0, nt), nt < 2^32 (32-bit trainIdx).  On
// success *tot holds the 128-row tiles the runs touch and the rows they hold; with `four` also the kRunFields layout of
// the device array (the host's own copy, for the planner's walk).
int check_runs(const int64_t* runs, long long n_runs, long long nt, RunTotals* tot, std::vector<long long>* four)
{
    if (n_runs < 0 || n_runs > 0x7FFFFFFFll || (n_runs > 0 && !runs)) {
        set_error("runs: bad count %lld or null host array", n_runs);
        return HM_ERR_INVALID_ARGUMENT;
    }
    if (nt < 0 || nt >= (1ll << 32)) {
        set_error("runs: train rows %lld outside [0, 2^32)", nt);
        return HM_ERR_INVALID_ARGUMENT;
    }
    long long prev = 0, tiles = 0, rows = 0;
    if (four) four->clear();
    for (long long i = 0; i < n_runs; ++i) {
        const long long lo = runs[2 * i], hi = runs[2 * i + 1];
        if (lo < prev || hi <= lo || hi > nt) {
            set_error("run %lld = [%lld, %lld): runs must be non-empty, ascending and disjoint within [0, %lld)", i, lo, hi,
                      nt);
            return HM_ERR_INVALID_ARGUMENT;
        }
        if (four) four->insert(four->end(), {lo, hi, tiles, rows});
        tiles += ceil_div(hi, 128) - lo / 128;
        rows += hi - lo;
        prev = hi;
    }
    if (tiles > 0x7FFFFFFFll) {
        set_error("runs: %lld tiles to walk", tiles);
        return HM_ERR_UNSUPPORTED;
    }
    tot->tiles = tiles;
    tot->rows = rows;
    return HM_OK;
}

int check_runs_dev(const int64_t* runs_dev, long long n_runs)
{
    if (n_runs > 0 && (!runs_dev || (reinterpret_cast<uintptr_t>(runs_dev) & 7))) {
        set_error("runs_dev: null or not 8-byte aligned");
        return HM_ERR_INVALID_ARGUMENT;
    }
    return HM_OK;
}

// hm_knn2_runs: [map: rows x u32 | gathered rows: rows x 32 B | workspace of hm_knn2 over the gathered rows]
size_t packed_runs_workspace(long long nq, long long rows, int variant, int sm_count)
{
    return align_up((size_t)rows * 4) + align_up((size_t)rows * HM_DESC_BYTES) + knn_workspace(nq, rows, 1, variant, sm_count);
}

// selected row j -> gathered[j] and map[j] = its shard-local row; one thread per 16 bytes.  The map ascends with j, so
// the stable order of the gathered problem is the stable order of the rows.
__global__ void hm_runs_gather_kernel(const uint8_t* train, long long t_stride, const long long* runs, int n_runs,
                                      long long rows, uint8_t* gathered, unsigned* map)
{
    const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= rows * 2) return;
    const long long j = o >> 1;
    int a = 0, b = n_runs - 1;                         // the last run whose row prefix is <= j
    while (a < b) {
        const int m = (a + b + 1) >> 1;
        if (runs[kRunFields * m + 3] <= j) a = m;
        else b = m - 1;
    }
    const long long row = runs[kRunFields * a] + (j - runs[kRunFields * a + 3]);
    reinterpret_cast<uint4*>(gathered)[o] = *reinterpret_cast<const uint4*>(train + row * t_stride + (o & 1) * 16);
    if (!(o & 1)) map[j] = (unsigned)row;
}

__global__ void hm_runs_remap_kernel(unsigned long long* keys, long long n, const unsigned* map,
                                     unsigned long long train_base)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned long long k = keys[i];
    if (k != kNoMatch) keys[i] = (k & 0xFFFFFFFF00000000ull) + train_base + map[k & 0xFFFFFFFFull];
}

}  // namespace
}  // namespace hm

using namespace hm;

extern "C" {

HM_API int hm_version(void) { return HM_ABI_VERSION; }

HM_API const char* hm_last_error(void) { return g_error; }

HM_API void hm_profile_events(void* start_event, void* stop_event)
{
    g_prof_start = static_cast<cudaEvent_t>(start_event);
    g_prof_stop = static_cast<cudaEvent_t>(stop_event);
    g_prof_armed = start_event && stop_event;
}

HM_API int hm_device_sm_count(void)
{
    DeviceInfo di;
    const int rc = device_info(&di);
    return rc == HM_OK ? di.sm_count : rc;
}

HM_API int hm_select_variant(int64_t nq, int64_t nt, int batch) { return select_variant(nq, nt, batch); }

HM_API int hm_describe_launch(int64_t nq, int64_t nt, int batch, int variant, char* buf, size_t buf_bytes)
{
    if (!buf || buf_bytes == 0 || nq <= 0 || nt <= 0 || batch <= 0) {
        set_error("hm_describe_launch: bad arguments");
        return HM_ERR_INVALID_ARGUMENT;
    }
    DeviceInfo di;
    int sm = 148;   // B200; the real count when a device is visible
    if (device_info(&di) == HM_OK) sm = di.sm_count;
    const int v = resolve_variant(variant, nq, nt, batch);
    if (v == HM_VARIANT_POPC) {
        KnnProblem p{};
        p.nq = nq; p.nt = nt; p.batch = batch;
        snprintf(buf, buf_bytes, "hm_popc_knn2_kernel splits=%d", popc_splits(p, sm));
    } else {
        describe_tc_launch(nq, nt, batch, sm, v, false, buf, buf_bytes);
    }
    return HM_OK;
}

HM_API size_t hm_workspace_bytes(int64_t nq, int64_t nt, int batch, int variant)
{
    DeviceInfo di;
    int sm = 148;   // sizing only; B200
    if (device_info(&di) == HM_OK) sm = di.sm_count;
    if (nq < 0 || nt < 0 || batch <= 0) return 0;
    // fused pipeline: fwd keys + bwd keys + the larger of the two k-NN passes
    const size_t fwd = align_up((size_t)batch * nq * 16);
    const size_t bwd = align_up((size_t)batch * nt * 16);
    const size_t a = knn_workspace(nq, nt, batch, variant, sm);
    const size_t b = knn_workspace(nt, nq, batch, variant, sm);
    return fwd + bwd + select_bytes(nt, batch) + (a > b ? a : b) + 256;
}

HM_API int hm_knn2(const uint8_t* query, int64_t nq, int64_t q_stride, const uint8_t* train, int64_t nt,
                   int64_t t_stride, uint64_t train_base, uint64_t* out_keys, int variant, void* workspace,
                   size_t workspace_bytes, void* stream)
{
    KnnProblem p{};
    p.q = query; p.t = train; p.nq = nq; p.nt = nt; p.q_stride = q_stride; p.t_stride = t_stride;
    p.batch = 1; p.train_base = train_base;
    return knn2_dispatch(p, reinterpret_cast<unsigned long long*>(out_keys), variant, workspace, workspace_bytes,
                         static_cast<cudaStream_t>(stream));
}

HM_API int hm_knn2_batched(const uint8_t* query, int64_t nq, int64_t q_stride, int64_t q_batch_stride,
                           const uint8_t* train, int64_t nt, int64_t t_stride, int64_t t_batch_stride, int batch,
                           uint64_t* out_keys, int variant, void* workspace, size_t workspace_bytes, void* stream)
{
    KnnProblem p{};
    p.q = query; p.t = train; p.nq = nq; p.nt = nt; p.q_stride = q_stride; p.t_stride = t_stride;
    p.q_batch_stride = q_batch_stride; p.t_batch_stride = t_batch_stride;
    p.batch = batch; p.train_base = 0;
    return knn2_dispatch(p, reinterpret_cast<unsigned long long*>(out_keys), variant, workspace, workspace_bytes,
                         static_cast<cudaStream_t>(stream));
}

HM_API int hm_default_tensor_variant(void) { return default_tensor_variant(); }

HM_API size_t hm_prepared_workspace_bytes(int64_t nq, int64_t nt, int variant)
{
    DeviceInfo di;
    int sm = 148;
    if (device_info(&di) == HM_OK) sm = di.sm_count;
    const int v = resolve_tensor_variant(variant);
    if (v < 0) return 0;
    if (nq <= 0 || nt <= 0) return 256;
    return align_up(tc_workspace_bytes(nq, nt, 1, sm, false, v));
}

HM_API size_t hm_prepared_bytes(int64_t n, int variant)
{
    const int v = resolve_tensor_variant(variant);
    return (n > 0 && v > 0) ? prepared_bytes(n, v) : 0;
}

HM_API int hm_prepare(const uint8_t* bits, int64_t n, int64_t stride, void* prepared, int variant, void* stream)
{
    DeviceInfo di;
    int rc = device_info(&di);
    if (rc != HM_OK) return rc;
    const int v = resolve_tensor_variant(variant);
    if (v < 0) return v;
    if ((rc = check_rows(bits, n, stride, "bits")) != HM_OK) return rc;
    if (n > 0 && (!prepared || (reinterpret_cast<uintptr_t>(prepared) & 15))) {
        set_error("prepared buffer must be non-null and 16-byte aligned");
        return HM_ERR_INVALID_ARGUMENT;
    }
    return launch_prepare(bits, n, stride, 0, 1, prepared, v, static_cast<cudaStream_t>(stream));
}

HM_API int hm_knn2_prepared(const void* query_prepared, int64_t nq, const void* train_prepared, int64_t nt,
                            uint64_t train_base, uint64_t* out_keys, int variant, void* workspace,
                            size_t workspace_bytes, void* stream)
{
    DeviceInfo di;
    int rc = device_info(&di);
    if (rc != HM_OK) return rc;
    const int v = resolve_tensor_variant(variant);
    if (v < 0) return v;
    if (nq < 0 || nt < 0) {
        set_error("negative row count");
        return HM_ERR_INVALID_ARGUMENT;
    }
    if (nq == 0) return HM_OK;
    if (!out_keys) {
        set_error("out_keys is null");
        return HM_ERR_INVALID_ARGUMENT;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (nt == 0) return fill_no_match(reinterpret_cast<unsigned long long*>(out_keys), nq * 2, st);
    if (!query_prepared || !train_prepared || (reinterpret_cast<uintptr_t>(query_prepared) & 15) ||
        (reinterpret_cast<uintptr_t>(train_prepared) & 15)) {
        set_error("prepared operands must be non-null and 16-byte aligned");
        return HM_ERR_INVALID_ARGUMENT;
    }
    return launch_tc_knn2_prepared(query_prepared, nq, train_prepared, nt, 1, train_base,
                                   reinterpret_cast<unsigned long long*>(out_keys), workspace, workspace_bytes,
                                   di.sm_count, v, st);
}

HM_API int hm_knn2_prepared_partials(const void* query_prepared, int64_t nq, const void* train_prepared, int64_t nt,
                                     uint64_t train_base, int variant, void* workspace, size_t workspace_bytes,
                                     void* stream, const uint64_t** out_partials, int* out_groups)
{
    DeviceInfo di;
    int rc = device_info(&di);
    if (rc != HM_OK) return rc;
    const int v = resolve_tensor_variant(variant);
    if (v < 0) return v;
    if (nq <= 0 || nt <= 0 || !out_partials || !out_groups || !query_prepared || !train_prepared) {
        set_error("hm_knn2_prepared_partials: bad arguments");
        return HM_ERR_INVALID_ARGUMENT;
    }
    const unsigned long long* parts = nullptr;
    rc = launch_tc_knn2_prepared(query_prepared, nq, train_prepared, nt, 1, train_base, nullptr, workspace,
                                 workspace_bytes, di.sm_count, v, static_cast<cudaStream_t>(stream), &parts, out_groups);
    *out_partials = reinterpret_cast<const uint64_t*>(parts);
    return rc;
}

HM_API int hm_knn2_prepared_exchange(const void* query_prepared, int64_t nq, const void* train_prepared, int64_t nt,
                                     uint64_t train_base, int world, int rank, void* const* peer_buffers_host,
                                     int64_t max_rows, uint32_t epoch, uint64_t* out_keys, int variant, void* workspace,
                                     size_t workspace_bytes, void* stream)
{
    DeviceInfo di;
    int rc = device_info(&di);
    if (rc != HM_OK) return rc;
    const int v = resolve_tensor_variant(variant);
    if (v < 0) return v;
    if (nq <= 0 || nt <= 0 || !out_keys || !query_prepared || !train_prepared) {
        set_error("hm_knn2_prepared_exchange: bad arguments");
        return HM_ERR_INVALID_ARGUMENT;
    }
    ExchangeArgs x;
    if ((rc = fill_exchange_args(&x, world, rank, peer_buffers_host, max_rows, epoch, nq)) != HM_OK) return rc;
    return launch_tc_knn2_prepared(query_prepared, nq, train_prepared, nt, 1, train_base,
                                   reinterpret_cast<unsigned long long*>(out_keys), workspace, workspace_bytes,
                                   di.sm_count, v, static_cast<cudaStream_t>(stream), nullptr, nullptr, &x);
}

HM_API size_t hm_resident_workspace_bytes(int64_t nq, int64_t nt, int variant)
{
    DeviceInfo di;
    int sm = 148;
    if (device_info(&di) == HM_OK) sm = di.sm_count;
    const int v = resolve_tensor_variant(variant);
    if (v < 0) return 0;
    if (nq <= 0 || nt <= 0) return 256;
    return align_up(tc_resident_workspace_bytes(nq, nt, sm, v));
}

static int knn2_resident_common(const uint8_t* query, int64_t nq, int64_t q_stride, const void* train_prepared, int64_t nt,
                                uint64_t train_base, uint64_t* out_keys, int variant, void* workspace,
                                size_t workspace_bytes, void* stream, const ExchangeArgs* x, const char* who)
{
    DeviceInfo di;
    int rc = device_info(&di);
    if (rc != HM_OK) return rc;
    const int v = resolve_tensor_variant(variant);
    if (v < 0) return v;
    if (nq < 0 || nt < 0) {
        set_error("%s: negative row count", who);
        return HM_ERR_INVALID_ARGUMENT;
    }
    if (nq == 0) return HM_OK;
    if (!out_keys) {
        set_error("%s: out_keys is null", who);
        return HM_ERR_INVALID_ARGUMENT;
    }
    if ((rc = check_rows(query, nq, q_stride, "query")) != HM_OK) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (nt == 0 && !x) return fill_no_match(reinterpret_cast<unsigned long long*>(out_keys), nq * 2, st);
    if (nt <= 0 || !train_prepared || (reinterpret_cast<uintptr_t>(train_prepared) & 15)) {
        set_error("%s: the prepared database must be non-empty, non-null and 16-byte aligned", who);
        return HM_ERR_INVALID_ARGUMENT;
    }
    return launch_tc_knn2_resident(query, nq, q_stride, train_prepared, nt, train_base,
                                   reinterpret_cast<unsigned long long*>(out_keys), workspace, workspace_bytes, di.sm_count,
                                   v, st, x);
}

HM_API int hm_knn2_resident(const uint8_t* query, int64_t nq, int64_t q_stride, const void* train_prepared, int64_t nt,
                            uint64_t train_base, uint64_t* out_keys, int variant, void* workspace,
                            size_t workspace_bytes, void* stream)
{
    return knn2_resident_common(query, nq, q_stride, train_prepared, nt, train_base, out_keys, variant, workspace,
                                workspace_bytes, stream, nullptr, "hm_knn2_resident");
}

HM_API int hm_knn2_resident_exchange(const uint8_t* query, int64_t nq, int64_t q_stride, const void* train_prepared,
                                     int64_t nt, uint64_t train_base, int world, int rank,
                                     void* const* peer_buffers_host, int64_t max_rows, uint32_t epoch, uint64_t* out_keys,
                                     int variant, void* workspace, size_t workspace_bytes, void* stream)
{
    ExchangeArgs x;
    DeviceInfo di;
    int rc = device_info(&di);
    if (rc != HM_OK) return rc;
    if (nq <= 0 || nt <= 0) {
        set_error("hm_knn2_resident_exchange: needs rows on both sides (every rank posts its flags)");
        return HM_ERR_INVALID_ARGUMENT;
    }
    if ((rc = fill_exchange_args(&x, world, rank, peer_buffers_host, max_rows, epoch, nq)) != HM_OK) return rc;
    return knn2_resident_common(query, nq, q_stride, train_prepared, nt, train_base, out_keys, variant, workspace,
                                workspace_bytes, stream, &x, "hm_knn2_resident_exchange");
}

HM_API size_t hm_runs_workspace_bytes(int64_t nq, const int64_t* runs_host, int64_t n_runs, int prepared, int variant)
{
    DeviceInfo di;
    int sm = 148;
    if (device_info(&di) == HM_OK) sm = di.sm_count;
    RunTotals tot;
    if (nq < 0 || check_runs(runs_host, n_runs, (1ll << 32) - 1, &tot, nullptr) != HM_OK) return 0;
    if (prepared) {
        const int v = resolve_tensor_variant(variant);
        if (v < 0) return 0;
        if (nq == 0 || tot.tiles == 0) return 256;
        return align_up(tc_resident_workspace_bytes(nq, tot.tiles * 128, sm, v));
    }
    if (variant < HM_VARIANT_AUTO || variant > HM_VARIANT_F4) return 0;
    if (nq == 0 || tot.rows == 0) return 256;
    return align_up(packed_runs_workspace(nq, tot.rows, variant, sm));
}

HM_API int hm_describe_runs_launch(int64_t nq, int64_t nt, const int64_t* runs_host, int64_t n_runs, int variant,
                                   char* buf, size_t buf_bytes, int64_t* pieces_host)
{
    if (nq <= 0) {
        set_error("hm_describe_runs_launch: needs query rows");
        return HM_ERR_INVALID_ARGUMENT;
    }
    const int v = resolve_tensor_variant(variant);
    if (v < 0) return v;
    RunTotals tot;
    std::vector<long long> four;
    const int rc = check_runs(runs_host, n_runs, nt, &tot, &four);
    if (rc != HM_OK) return rc;
    if (n_runs == 0) {
        if (buf && buf_bytes) snprintf(buf, buf_bytes, "no launch: empty selection");
        return 0;
    }
    DeviceInfo di;
    int sm = 148;   // B200; the real count when a device is visible
    if (device_info(&di) == HM_OK) sm = di.sm_count;
    describe_tc_runs(nq, four.data(), (int)n_runs, tot.tiles, sm, v, buf, buf_bytes,
                     reinterpret_cast<long long*>(pieces_host));
    return (int)tot.tiles;
}

static int knn2_resident_runs_common(const uint8_t* query, int64_t nq, int64_t q_stride, const void* train_prepared,
                                     int64_t nt, const int64_t* runs_host, const int64_t* runs_dev, int64_t n_runs,
                                     uint64_t train_base, uint64_t* out_keys, int variant, void* workspace,
                                     size_t workspace_bytes, void* stream, const ExchangeArgs* x, const char* who)
{
    DeviceInfo di;
    int rc = device_info(&di);
    if (rc != HM_OK) return rc;
    const int v = resolve_tensor_variant(variant);
    if (v < 0) return v;
    RunTotals tot;
    if ((rc = check_runs(runs_host, n_runs, nt, &tot, nullptr)) != HM_OK) return rc;
    if ((rc = check_runs_dev(runs_dev, n_runs)) != HM_OK) return rc;
    if (nq < 0) {
        set_error("%s: negative row count", who);
        return HM_ERR_INVALID_ARGUMENT;
    }
    if (nq == 0) return HM_OK;
    if (!out_keys) {
        set_error("%s: out_keys is null", who);
        return HM_ERR_INVALID_ARGUMENT;
    }
    if ((rc = check_rows(query, nq, q_stride, "query")) != HM_OK) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (n_runs == 0) {
        if (x) {
            set_error("%s: needs at least one run (a rank without selected rows joins through hm_exchange_merge)", who);
            return HM_ERR_INVALID_ARGUMENT;
        }
        return fill_no_match(reinterpret_cast<unsigned long long*>(out_keys), nq * 2, st);
    }
    if (!train_prepared || (reinterpret_cast<uintptr_t>(train_prepared) & 15)) {
        set_error("%s: the prepared database must be non-null and 16-byte aligned", who);
        return HM_ERR_INVALID_ARGUMENT;
    }
    const RunArgs ra{reinterpret_cast<const long long*>(runs_dev), (int)n_runs};
    return launch_tc_knn2_resident_runs(query, nq, q_stride, train_prepared, nt, ra, tot, train_base,
                                        reinterpret_cast<unsigned long long*>(out_keys), workspace, workspace_bytes,
                                        di.sm_count, v, st, x);
}

HM_API int hm_knn2_resident_runs(const uint8_t* query, int64_t nq, int64_t q_stride, const void* train_prepared,
                                 int64_t nt, const int64_t* runs_host, const int64_t* runs_dev, int64_t n_runs,
                                 uint64_t train_base, uint64_t* out_keys, int variant, void* workspace,
                                 size_t workspace_bytes, void* stream)
{
    return knn2_resident_runs_common(query, nq, q_stride, train_prepared, nt, runs_host, runs_dev, n_runs, train_base,
                                     out_keys, variant, workspace, workspace_bytes, stream, nullptr,
                                     "hm_knn2_resident_runs");
}

HM_API int hm_knn2_resident_runs_exchange(const uint8_t* query, int64_t nq, int64_t q_stride, const void* train_prepared,
                                          int64_t nt, const int64_t* runs_host, const int64_t* runs_dev, int64_t n_runs,
                                          uint64_t train_base, int world, int rank, void* const* peer_buffers_host,
                                          int64_t max_rows, uint32_t epoch, uint64_t* out_keys, int variant,
                                          void* workspace, size_t workspace_bytes, void* stream)
{
    ExchangeArgs x;
    DeviceInfo di;
    int rc = device_info(&di);
    if (rc != HM_OK) return rc;
    if (nq <= 0) {
        set_error("hm_knn2_resident_runs_exchange: needs query rows (every rank posts its flags)");
        return HM_ERR_INVALID_ARGUMENT;
    }
    if ((rc = fill_exchange_args(&x, world, rank, peer_buffers_host, max_rows, epoch, nq)) != HM_OK) return rc;
    return knn2_resident_runs_common(query, nq, q_stride, train_prepared, nt, runs_host, runs_dev, n_runs, train_base,
                                     out_keys, variant, workspace, workspace_bytes, stream, &x,
                                     "hm_knn2_resident_runs_exchange");
}

HM_API int hm_knn2_runs(const uint8_t* query, int64_t nq, int64_t q_stride, const uint8_t* train, int64_t nt,
                        int64_t t_stride, const int64_t* runs_host, const int64_t* runs_dev, int64_t n_runs,
                        uint64_t train_base, uint64_t* out_keys, int variant, void* workspace, size_t workspace_bytes,
                        void* stream)
{
    DeviceInfo di;
    int rc = device_info(&di);
    if (rc != HM_OK) return rc;
    if (variant < HM_VARIANT_AUTO || variant > HM_VARIANT_F4) {
        set_error("unknown variant %d", variant);
        return HM_ERR_INVALID_ARGUMENT;
    }
    RunTotals tot;
    if ((rc = check_runs(runs_host, n_runs, nt, &tot, nullptr)) != HM_OK) return rc;
    if ((rc = check_runs_dev(runs_dev, n_runs)) != HM_OK) return rc;
    if (nq < 0) {
        set_error("hm_knn2_runs: negative row count");
        return HM_ERR_INVALID_ARGUMENT;
    }
    if (nq == 0) return HM_OK;
    if (!out_keys) {
        set_error("hm_knn2_runs: out_keys is null");
        return HM_ERR_INVALID_ARGUMENT;
    }
    if ((rc = check_rows(query, nq, q_stride, "query")) != HM_OK) return rc;
    if ((rc = check_rows(train, nt, t_stride, "train")) != HM_OK) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    unsigned long long* out = reinterpret_cast<unsigned long long*>(out_keys);
    if (tot.rows == 0) return fill_no_match(out, nq * 2, st);
    const size_t need = packed_runs_workspace(nq, tot.rows, variant, di.sm_count);
    if (!workspace || workspace_bytes < need) {
        set_error("workspace too small: need %zu bytes, got %zu", need, workspace_bytes);
        return HM_ERR_WORKSPACE;
    }
    unsigned* map = static_cast<unsigned*>(workspace);
    uint8_t* gathered = static_cast<uint8_t*>(workspace) + align_up((size_t)tot.rows * 4);
    const size_t head = align_up((size_t)tot.rows * 4) + align_up((size_t)tot.rows * HM_DESC_BYTES);
    hm_runs_gather_kernel<<<(unsigned)ceil_div(tot.rows * 2, 256), 256, 0, st>>>(
        train, t_stride, reinterpret_cast<const long long*>(runs_dev), (int)n_runs, tot.rows, gathered, map);
    HM_CUDA_CHECK(cudaGetLastError());
    KnnProblem p{};
    p.q = query; p.t = gathered; p.nq = nq; p.nt = tot.rows; p.q_stride = q_stride; p.t_stride = HM_DESC_BYTES;
    p.batch = 1; p.train_base = 0;
    if ((rc = knn2_dispatch(p, out, variant, static_cast<uint8_t*>(workspace) + head, workspace_bytes - head, st)) != HM_OK)
        return rc;
    hm_runs_remap_kernel<<<(unsigned)ceil_div(nq * 2, 256), 256, 0, st>>>(out, nq * 2, map, train_base);
    HM_CUDA_CHECK(cudaGetLastError());
    return HM_OK;
}

HM_API int hm_merge_top2(const uint64_t* keys, int groups, int64_t rows, uint64_t* out_keys, void* stream)
{
    DeviceInfo di;
    int rc = device_info(&di);
    if (rc != HM_OK) return rc;
    if (groups <= 0 || rows < 0 || (rows > 0 && (!keys || !out_keys))) {
        set_error("hm_merge_top2: bad arguments");
        return HM_ERR_INVALID_ARGUMENT;
    }
    return launch_merge_top2(reinterpret_cast<const unsigned long long*>(keys), groups, rows,
                             reinterpret_cast<unsigned long long*>(out_keys), static_cast<cudaStream_t>(stream));
}

HM_API size_t hm_exchange_bytes(int64_t max_rows, int world)
{
    if (max_rows <= 0 || world < 1 || world > kMaxWorld) return 0;
    return exchange_bytes(max_rows, world);
}

HM_API int hm_exchange_merge(const uint64_t* local_keys, int local_groups, int64_t rows, int world, int rank,
                             void* const* peer_buffers_host, int64_t max_rows, uint32_t epoch, uint64_t* out_keys,
                             void* stream)
{
    DeviceInfo di;
    int rc = device_info(&di);
    if (rc != HM_OK) return rc;
    if (!local_keys || !out_keys || !peer_buffers_host) {
        set_error("hm_exchange_merge: null pointer");
        return HM_ERR_INVALID_ARGUMENT;
    }
    return launch_exchange_merge(reinterpret_cast<const unsigned long long*>(local_keys), local_groups, rows, world, rank,
                                 peer_buffers_host, max_rows, epoch, reinterpret_cast<unsigned long long*>(out_keys),
                                 static_cast<cudaStream_t>(stream));
}

static int build_filter_args(unsigned flags, const uint16_t* ratio_lut_host, double dist_threshold, RatioLut* lut,
                             int* thr_ceil)
{
    memset(lut, 0, sizeof(*lut));
    if (flags & HM_FLAG_RATIO) {
        if (!ratio_lut_host) {
            set_error("HM_FLAG_RATIO needs ratio_lut_host[257]");
            return HM_ERR_INVALID_ARGUMENT;
        }
        memcpy(lut->v, ratio_lut_host, sizeof(lut->v));
    }
    *thr_ceil = 0;
    if (flags & HM_FLAG_DIST_THRESHOLD) {
        // integer d < x  <=>  d < ceil(x): exact form of the reference's float compare
        double c = ceil(dist_threshold);
        if (!(c == c)) c = 0;                 // NaN compares false everywhere
        if (c > 1e9) c = 1e9;
        if (c < -1e9) c = -1e9;
        *thr_ceil = (int)c;
    }
    return HM_OK;
}

HM_API int hm_filter_matches(const uint64_t* fwd_keys, int64_t nq, const uint64_t* bwd_keys, int64_t nt, int batch,
                             unsigned flags, const uint16_t* ratio_lut_host, double dist_threshold, int32_t* out_q,
                             int32_t* out_t, int32_t* out_d, int32_t* out_count, void* stream)
{
    DeviceInfo di;
    int rc = device_info(&di);
    if (rc != HM_OK) return rc;
    if (batch <= 0) return HM_OK;
    if (nq < 0 || nt < 0 || !out_count || (nq > 0 && (!fwd_keys || !out_q || !out_t || !out_d)) ||
        ((flags & HM_FLAG_MUTUAL) && nt > 0 && !bwd_keys)) {
        set_error("hm_filter_matches: bad arguments");
        return HM_ERR_INVALID_ARGUMENT;
    }
    RatioLut lut;
    int thr;
    if ((rc = build_filter_args(flags, ratio_lut_host, dist_threshold, &lut, &thr)) != HM_OK) return rc;
    return launch_filter(reinterpret_cast<const unsigned long long*>(fwd_keys), nq,
                         reinterpret_cast<const unsigned long long*>(bwd_keys), nt, batch, flags, lut, thr, out_q,
                         out_t, out_d, out_count, static_cast<cudaStream_t>(stream));
}

HM_API int hm_match_fused(const uint8_t* query, int64_t nq, int64_t q_stride, int64_t q_batch_stride,
                          const uint8_t* train, int64_t nt, int64_t t_stride, int64_t t_batch_stride, int batch,
                          unsigned flags, const uint16_t* ratio_lut_host, double dist_threshold, int32_t* out_q,
                          int32_t* out_t, int32_t* out_d, int32_t* out_count, uint64_t* out_keys, int variant,
                          void* workspace, size_t workspace_bytes, void* stream)
{
    DeviceInfo di;
    int rc = device_info(&di);
    if (rc != HM_OK) return rc;
    if (batch <= 0) return HM_OK;
    if (!out_count || (nq > 0 && (!out_q || !out_t || !out_d))) {      // before anything is enqueued
        set_error("hm_match_fused: null output");
        return HM_ERR_INVALID_ARGUMENT;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    RatioLut lut;
    int thr;
    if ((rc = build_filter_args(flags, ratio_lut_host, dist_threshold, &lut, &thr)) != HM_OK) return rc;
    const size_t need = hm_workspace_bytes(nq, nt, batch, variant);
    if (!workspace || workspace_bytes < need) {
        set_error("workspace too small: need %zu bytes, got %zu", need, workspace_bytes);
        return HM_ERR_WORKSPACE;
    }
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    const size_t fwd_bytes = align_up((size_t)batch * nq * 16);
    const size_t bwd_bytes = align_up((size_t)batch * nt * 16);
    unsigned long long* fwd = out_keys ? reinterpret_cast<unsigned long long*>(out_keys)
                                       : reinterpret_cast<unsigned long long*>(ws);
    unsigned long long* bwd = reinterpret_cast<unsigned long long*>(ws + fwd_bytes);
    uint8_t* sel_ws = ws + fwd_bytes + bwd_bytes;
    const size_t sel_bytes = select_bytes(nt, batch);
    uint8_t* knn_ws = sel_ws + sel_bytes;
    const size_t knn_ws_bytes = workspace_bytes - fwd_bytes - bwd_bytes - sel_bytes;

    KnnProblem p{};
    p.q = query; p.t = train; p.nq = nq; p.nt = nt; p.q_stride = q_stride; p.t_stride = t_stride;
    p.q_batch_stride = q_batch_stride; p.t_batch_stride = t_batch_stride; p.batch = batch;
    // cv2.BFMatcher.match() -- the reference's own call (feature_matchers.py:39) -- is k = 1: without the ratio
    // test nobody reads the second neighbour
    p.top1 = !(flags & HM_FLAG_RATIO) && !out_keys;
    const bool mutual = (flags & HM_FLAG_MUTUAL) && nq > 0 && nt > 0;
    // Mutual check with the kind::mxf4 core: the forward kernel applies the ratio test to each row's final keys and
    // marks the best train row of every survivor as a candidate; the swapped pass then computes the best query of the
    // CANDIDATE train rows only (gathered inside the kernel from a device-side list).  A match (q, t) is mutual iff q
    // is the best query of t, and only candidates are ever asked -- same result as the full swapped pass, for the
    // fraction of its work that the ratio test leaves.
    if (mutual && resolve_variant(variant, nq, nt, batch) == HM_VARIANT_F4) {
        SelectArgs sel;
        memset(&sel, 0, sizeof(sel));
        sel.count = reinterpret_cast<int*>(sel_ws);
        sel.slot_of = reinterpret_cast<int*>(sel_ws + align_up((size_t)batch * 4));
        sel.list = reinterpret_cast<int*>(sel_ws + select_zeroed_bytes(nt, batch));
        sel.nt = nt;
        sel.use_ratio = (flags & HM_FLAG_RATIO) ? 1 : 0;
        sel.lut = lut;
        HM_CUDA_CHECK(cudaMemsetAsync(sel_ws, 0, select_zeroed_bytes(nt, batch), st));
        p.select = &sel;
        if ((rc = knn2_dispatch(p, fwd, HM_VARIANT_F4, knn_ws, knn_ws_bytes, st)) != HM_OK) return rc;
        KnnProblem r{};
        r.q = train; r.t = query; r.nq = nt; r.nt = nq; r.q_stride = t_stride; r.t_stride = q_stride;
        r.q_batch_stride = t_batch_stride; r.t_batch_stride = q_batch_stride; r.batch = batch;
        r.top1 = true;
        if ((rc = launch_tc_knn1_candidates(r, sel.list, sel.count, bwd, knn_ws, knn_ws_bytes, di.sm_count, st)) != HM_OK) return rc;
        return launch_filter(fwd, nq, bwd, nt, batch, flags, lut, thr, out_q, out_t, out_d, out_count, st, sel.slot_of);
    }
    if ((rc = knn2_dispatch(p, fwd, variant, knn_ws, knn_ws_bytes, st)) != HM_OK) return rc;
    if (mutual) {
        KnnProblem r{};
        r.q = train; r.t = query; r.nq = nt; r.nt = nq; r.q_stride = t_stride; r.t_stride = q_stride;
        r.q_batch_stride = t_batch_stride; r.t_batch_stride = q_batch_stride; r.batch = batch;
        r.top1 = true;                       // the filter only reads each train row's best query
        if ((rc = knn2_dispatch(r, bwd, variant, knn_ws, knn_ws_bytes, st)) != HM_OK) return rc;
    }
    return launch_filter(fwd, nq, bwd, nt, batch, flags, lut, thr, out_q, out_t, out_d, out_count, st);
}

// ---- keyframe database: ratio test + database-wide mutual check ----------------------------------------------------
// Workspace of hm_db_mutual_flags, all sized by the query batch alone: [count | list nq | owner nq | best nq x 2 |
// gathered rows nq x 32 | k-NN scratch of the nq x nq top-1 pass].  `v` is the variant resolved for nq x nq.
struct DbMutualLayout {
    size_t list, owner, best, gathered, knn, total;
};

static DbMutualLayout db_mutual_layout(long long nq, int v, int sm)
{
    DbMutualLayout L;
    L.list = 256;
    L.owner = L.list + align_up((size_t)nq * 4);
    L.best = L.owner + align_up((size_t)nq * 4);
    L.gathered = L.best + align_up((size_t)nq * 16);
    L.knn = L.gathered + align_up((size_t)nq * HM_DESC_BYTES);
    // kind::mxf4 runs the candidate pass (the kernel gathers the rows through the list); the other cores a dense pass
    // over the gathered rows
    const size_t k = v == HM_VARIANT_F4 ? tc_workspace_bytes(nq, nq, 1, sm, true, HM_VARIANT_F4) : knn_workspace(nq, nq, 1, v, sm);
    L.total = L.knn + align_up(k) + 256;
    return L;
}

HM_API size_t hm_db_mutual_workspace_bytes(int64_t nq, int variant)
{
    DeviceInfo di;
    int sm = 148;   // sizing only; B200
    if (device_info(&di) == HM_OK) sm = di.sm_count;
    if (nq < 0 || variant < HM_VARIANT_AUTO || variant > HM_VARIANT_F4) return 0;
    if (nq == 0) return 256;
    return db_mutual_layout(nq, resolve_variant(variant, nq, nq, 1), sm).total;
}

HM_API int hm_db_mutual_flags(const uint64_t* keys, int64_t nq, const uint8_t* query, int64_t q_stride,
                              const uint8_t* shard_bits, int64_t shard_rows, int64_t t_stride, uint64_t row_lo,
                              unsigned flags, const uint16_t* ratio_lut_host, uint8_t* out_flags, int variant,
                              void* workspace, size_t workspace_bytes, void* stream)
{
    DeviceInfo di;
    int rc = device_info(&di);
    if (rc != HM_OK) return rc;
    if (nq < 0 || shard_rows < 0 || (nq > 0 && (!keys || !out_flags)) || (flags & ~(HM_FLAG_RATIO | HM_FLAG_MUTUAL)) ||
        variant < HM_VARIANT_AUTO || variant > HM_VARIANT_F4 || row_lo + (uint64_t)shard_rows > 0xFFFFFFFFull) {
        set_error("hm_db_mutual_flags: bad arguments");
        return HM_ERR_INVALID_ARGUMENT;
    }
    if (nq == 0) return HM_OK;
    if ((rc = check_rows(query, nq, q_stride, "query")) != HM_OK) return rc;
    if ((rc = check_rows(shard_bits, shard_rows, t_stride, "shard_bits")) != HM_OK) return rc;
    RatioLut lut;
    int thr;
    if ((rc = build_filter_args(flags & HM_FLAG_RATIO, ratio_lut_host, 0.0, &lut, &thr)) != HM_OK) return rc;
    const int v = resolve_variant(variant, nq, nq, 1);
    const DbMutualLayout L = db_mutual_layout(nq, v, di.sm_count);
    if (!workspace || workspace_bytes < L.total || (reinterpret_cast<uintptr_t>(workspace) & 255)) {
        set_error("workspace too small or misaligned: need %zu bytes, 256-byte aligned, got %zu", L.total, workspace_bytes);
        return HM_ERR_WORKSPACE;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    int* count = reinterpret_cast<int*>(ws);
    int* list = reinterpret_cast<int*>(ws + L.list);
    int* owner = reinterpret_cast<int*>(ws + L.owner);
    unsigned long long* best = reinterpret_cast<unsigned long long*>(ws + L.best);
    uint8_t* gathered = v == HM_VARIANT_F4 ? nullptr : ws + L.gathered;
    unsigned char* fl = reinterpret_cast<unsigned char*>(out_flags);
    const unsigned long long* k = reinterpret_cast<const unsigned long long*>(keys);
    // every flag is written (0) here, also on a shard without rows: the MAX over the shards needs each one's zeros
    if ((rc = launch_db_select(k, nq, row_lo, row_lo + (uint64_t)shard_rows, (flags & HM_FLAG_RATIO) ? 1 : 0, lut,
                               shard_bits, t_stride, list, owner, count, gathered, fl, st)) != HM_OK)
        return rc;
    if (shard_rows == 0) return HM_OK;
    // top-1 over the query batch of every listed shard row: "query" side = shard rows, "train" side = the batch
    KnnProblem r{};
    r.q = gathered ? gathered : shard_bits; r.nq = nq; r.q_stride = gathered ? HM_DESC_BYTES : t_stride;
    r.t = query; r.nt = nq; r.t_stride = q_stride;
    r.batch = 1; r.top1 = true;
    uint8_t* knn_ws = ws + L.knn;
    const size_t knn_bytes = L.total - L.knn;
    if (v == HM_VARIANT_F4) rc = launch_tc_knn1_candidates(r, list, count, best, knn_ws, knn_bytes, di.sm_count, st);
    else                    rc = knn2_dispatch(r, best, v, knn_ws, knn_bytes, st);
    if (rc != HM_OK) return rc;
    return launch_db_resolve(owner, count, best, nq, fl, st);
}

HM_API int hm_db_filter(const uint64_t* keys, int64_t nq, const uint8_t* mutual_flags, unsigned flags,
                        const uint16_t* ratio_lut_host, int32_t* out_q, int32_t* out_t, int32_t* out_d, int32_t* out_count,
                        void* stream)
{
    DeviceInfo di;
    int rc = device_info(&di);
    if (rc != HM_OK) return rc;
    if (nq < 0 || !out_count || (nq > 0 && (!keys || !out_q || !out_t || !out_d)) ||
        (flags & ~(HM_FLAG_RATIO | HM_FLAG_MUTUAL)) || ((flags & HM_FLAG_MUTUAL) && nq > 0 && !mutual_flags)) {
        set_error("hm_db_filter: bad arguments");
        return HM_ERR_INVALID_ARGUMENT;
    }
    RatioLut lut;
    int thr;
    if ((rc = build_filter_args(flags, ratio_lut_host, 0.0, &lut, &thr)) != HM_OK) return rc;
    return launch_filter(reinterpret_cast<const unsigned long long*>(keys), nq, nullptr, 0, 1, flags, lut, thr, out_q,
                         out_t, out_d, out_count, static_cast<cudaStream_t>(stream), nullptr,
                         reinterpret_cast<const unsigned char*>(mutual_flags));
}

HM_API int hm_gather_points(const int32_t* q_idx, const int32_t* t_idx, const int32_t* count, int64_t stride, int batch,
                            const int32_t* query_pts, int64_t nq, const int32_t* train_pts, int64_t nt,
                            int32_t* out_query_pts, int32_t* out_train_pts, void* stream)
{
    DeviceInfo di;
    int rc = device_info(&di);
    if (rc != HM_OK) return rc;
    if (batch <= 0 || stride <= 0) return HM_OK;
    if (!q_idx || !t_idx || !count || !query_pts || !train_pts || !out_query_pts || !out_train_pts || nq <= 0 || nt <= 0 ||
        ((reinterpret_cast<uintptr_t>(query_pts) | reinterpret_cast<uintptr_t>(train_pts) |
          reinterpret_cast<uintptr_t>(out_query_pts) | reinterpret_cast<uintptr_t>(out_train_pts)) & 7)) {
        set_error("hm_gather_points: null, empty or misaligned argument");
        return HM_ERR_INVALID_ARGUMENT;
    }
    return launch_gather_points(q_idx, t_idx, count, stride, batch, query_pts, nq, train_pts, nt, out_query_pts,
                                out_train_pts, static_cast<cudaStream_t>(stream));
}

HM_API int hm_rasterize_mask(const int32_t* points, int64_t n, int radius, int inner, uint8_t* mask, int h, int w,
                             int64_t row_stride, void* stream)
{
    DeviceInfo di;
    int rc = device_info(&di);
    if (rc != HM_OK) return rc;
    if (h < 0 || w < 0 || n < 0 || radius < 0 || ((h > 0 && w > 0) && (!mask || row_stride < w)) ||
        (n > 0 && (!points || (reinterpret_cast<uintptr_t>(points) & 7)))) {
        set_error("hm_rasterize_mask: bad arguments");
        return HM_ERR_INVALID_ARGUMENT;
    }
    return launch_rasterize_mask(points, n, radius, inner, mask, h, w, row_stride, static_cast<cudaStream_t>(stream));
}

// ---- host-buffer convenience ---------------------------------------------------------------
constexpr int kFrameSlots = HM_FRAME_SLOTS;

struct FrameSlot {
    uint8_t* d;          // device: [descriptors n x 32 | pad | positions n x 2 int32]
    size_t cap;
    int64_t n;
    bool has_points;
    uint8_t* h;          // pinned staging of this slot, same carving
    size_t h_cap;
    cudaEvent_t uploaded;   // the last H2D out of `h` (the next put into this slot waits for it)
};

// Small problems are bound by launch latency, not by the kernels (200 x 200: ~6 us of GPU work behind five
// driver calls): the host-buffer entry points replay a CUDA graph of their whole stream sequence -- H2D,
// memset, k-NN, filter, (gather,) D2H -- once a shape has been seen twice.
struct GraphKey {
    int kind;                        // 0 = hm_match_host, 1 = hm_frame_match
    int64_t nq, nt;
    unsigned flags;
    int variant, want_pts, has_lut;
    double thr;
    const void* ptr[4];              // every buffer the captured sequence touches
    uint16_t lut[257];
};

struct GraphEntry {
    GraphKey key;
    int uses;                        // calls seen with this key; -1 = capture failed, never try again
    cudaGraphExec_t exec;
};

constexpr int kGraphCache = 12;
constexpr double kGraphMaxPairs = 6.4e7;   // above this the launches are noise

struct hm_context {
    GraphEntry graphs[kGraphCache];
    int graph_next;
    cudaStream_t stream;
    uint8_t* d_buf;      // device: [query | train | keys | workspace]
    size_t d_cap;
    uint8_t* h_buf;      // pinned staging, same carving for query | train | keys
    size_t h_cap;
    FrameSlot slots[kFrameSlots];   // resident frames (hm_frame_put / hm_frame_match)
    cudaEvent_t staged;             // the last unsynchronised H2D out of h_buf (hm_frame_put_orb)
    unsigned small_epoch;           // call counter of the single-launch small-problem path (hm_small.cu)
};

HM_API int hm_context_create(hm_context** out_ctx)
{
    if (!out_ctx) {
        set_error("out_ctx is null");
        return HM_ERR_INVALID_ARGUMENT;
    }
    DeviceInfo di;
    int rc = device_info(&di);
    if (rc != HM_OK) return rc;
    hm_context* c = new (std::nothrow) hm_context();
    if (!c) {
        set_error("out of host memory");
        return HM_ERR_CUDA;
    }
    memset(c, 0, sizeof(*c));
    cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        set_error("cudaStreamCreate failed: %s", cudaGetErrorString(e));
        delete c;
        return HM_ERR_CUDA;
    }
    *out_ctx = c;
    return HM_OK;
}

HM_API void hm_context_destroy(hm_context* ctx)
{
    if (!ctx) return;
    for (GraphEntry& g : ctx->graphs)
        if (g.exec) cudaGraphExecDestroy(g.exec);
    for (FrameSlot& f : ctx->slots) {
        if (f.d) cudaFree(f.d);
        if (f.h) cudaFreeHost(f.h);
        if (f.uploaded) cudaEventDestroy(f.uploaded);
    }
    if (ctx->d_buf) cudaFree(ctx->d_buf);
    if (ctx->h_buf) cudaFreeHost(ctx->h_buf);
    if (ctx->staged) cudaEventDestroy(ctx->staged);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

}  // extern "C"

static bool same_key(const GraphKey& a, const GraphKey& b)
{
    return a.kind == b.kind && a.nq == b.nq && a.nt == b.nt && a.flags == b.flags && a.variant == b.variant &&
           a.want_pts == b.want_pts && a.has_lut == b.has_lut && a.thr == b.thr &&
           !memcmp(a.ptr, b.ptr, sizeof(a.ptr)) && (!a.has_lut || !memcmp(a.lut, b.lut, sizeof(a.lut)));
}

// Runs `enqueue()` (which only enqueues work on ctx->stream) directly the first time a key is seen, captures
// it into a graph the second time, and replays the graph afterwards.
template <class F>
static int run_cached_graph(hm_context* ctx, const GraphKey& key, F&& enqueue)
{
    const bool eligible = (double)key.nq * (double)key.nt <= kGraphMaxPairs && !(g_prof_start && g_prof_stop);
    if (!eligible) return enqueue();
    GraphEntry* e = nullptr;
    for (GraphEntry& g : ctx->graphs)
        if (g.uses != 0 && same_key(g.key, key)) { e = &g; break; }
    if (!e) {                                        // first sighting: run directly, remember the key
        e = &ctx->graphs[ctx->graph_next];
        ctx->graph_next = (ctx->graph_next + 1) % kGraphCache;
        if (e->exec) cudaGraphExecDestroy(e->exec);
        e->exec = nullptr;
        e->key = key;
        e->uses = 1;
        return enqueue();
    }
    if (e->uses < 0) return enqueue();
    if (!e->exec) {
        cudaGraph_t graph = nullptr;
        if (cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
            cudaGetLastError();
            e->uses = -1;
            return enqueue();
        }
        const int rc = enqueue();
        const cudaError_t ce = cudaStreamEndCapture(ctx->stream, &graph);
        if (rc != HM_OK || ce != cudaSuccess || !graph ||
            cudaGraphInstantiate(&e->exec, graph, 0) != cudaSuccess) {
            cudaGetLastError();
            if (graph) cudaGraphDestroy(graph);
            e->exec = nullptr;
            e->uses = -1;
            return enqueue();                        // nothing ran during the failed capture: run it directly
        }
        cudaGraphDestroy(graph);
    }
    ++e->uses;
    HM_CUDA_CHECK(cudaGraphLaunch(e->exec, ctx->stream));
    return HM_OK;
}

static void fill_key(GraphKey* k, int kind, int64_t nq, int64_t nt, unsigned flags, int variant, int want_pts,
                     const uint16_t* lut, double thr)
{
    memset(k, 0, sizeof(*k));
    k->kind = kind; k->nq = nq; k->nt = nt; k->flags = flags; k->variant = variant; k->want_pts = want_pts;
    k->thr = (flags & HM_FLAG_DIST_THRESHOLD) ? thr : 0.0;
    k->has_lut = (flags & HM_FLAG_RATIO) && lut;
    if (k->has_lut) memcpy(k->lut, lut, sizeof(k->lut));
}

extern "C" {

HM_API int hm_knn2_host(hm_context* ctx, const uint8_t* query_host, int64_t nq, const uint8_t* train_host, int64_t nt,
                        uint64_t* out_keys_host, int variant)
{
    if (!ctx || nq < 0 || nt < 0 || (nq > 0 && (!query_host || !out_keys_host)) || (nt > 0 && !train_host)) {
        set_error("hm_knn2_host: bad arguments");
        return HM_ERR_INVALID_ARGUMENT;
    }
    if (nq == 0) return HM_OK;
    const size_t qb = align_up((size_t)nq * HM_DESC_BYTES, 1024), tb = align_up((size_t)nt * HM_DESC_BYTES, 1024);
    const size_t kb = align_up((size_t)nq * 16, 1024);
    const size_t wsb = align_up(hm_workspace_bytes(nq, nt, 1, variant), 1024);
    const size_t dneed = qb + tb + kb + wsb, hneed = qb + tb + kb;
    if (ctx->staged) HM_CUDA_CHECK(cudaEventSynchronize(ctx->staged));      // see ctx_reserve
    if (ctx->d_cap < dneed || ctx->h_cap < hneed) HM_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    if (ctx->d_cap < dneed) {
        if (ctx->d_buf) cudaFree(ctx->d_buf);
        ctx->d_buf = nullptr; ctx->d_cap = 0;
        HM_CUDA_CHECK(cudaMalloc(&ctx->d_buf, dneed));
        ctx->d_cap = dneed;
    }
    if (ctx->h_cap < hneed) {
        if (ctx->h_buf) cudaFreeHost(ctx->h_buf);
        ctx->h_buf = nullptr; ctx->h_cap = 0;
        HM_CUDA_CHECK(cudaMallocHost(&ctx->h_buf, hneed));
        ctx->h_cap = hneed;
    }
    uint8_t *dq = ctx->d_buf, *dt = dq + qb, *dk = dt + tb, *dw = dk + kb;
    uint8_t *hq = ctx->h_buf, *ht = hq + qb, *hk = ht + tb;
    memcpy(hq, query_host, (size_t)nq * HM_DESC_BYTES);
    if (nt) memcpy(ht, train_host, (size_t)nt * HM_DESC_BYTES);
    HM_CUDA_CHECK(cudaMemcpyAsync(dq, hq, (size_t)nq * HM_DESC_BYTES, cudaMemcpyHostToDevice, ctx->stream));
    if (nt) HM_CUDA_CHECK(cudaMemcpyAsync(dt, ht, (size_t)nt * HM_DESC_BYTES, cudaMemcpyHostToDevice, ctx->stream));
    int rc = hm_knn2(dq, nq, HM_DESC_BYTES, dt, nt, HM_DESC_BYTES, 0, reinterpret_cast<uint64_t*>(dk), variant, dw, wsb,
                     ctx->stream);
    if (rc != HM_OK) return rc;
    HM_CUDA_CHECK(cudaMemcpyAsync(hk, dk, (size_t)nq * 16, cudaMemcpyDeviceToHost, ctx->stream));
    HM_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    memcpy(out_keys_host, hk, (size_t)nq * 16);
    return HM_OK;
}

static int ctx_reserve(hm_context* ctx, size_t dneed, size_t hneed)
{
    // every caller is about to overwrite h_buf: an unsynchronised upload out of it (hm_frame_put_orb) must have left
    if (ctx->staged) HM_CUDA_CHECK(cudaEventSynchronize(ctx->staged));
    if (ctx->d_cap < dneed || ctx->h_cap < hneed) HM_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));   // queued work may still use the old buffers
    if (ctx->d_cap < dneed) {
        if (ctx->d_buf) cudaFree(ctx->d_buf);
        ctx->d_buf = nullptr; ctx->d_cap = 0;
        HM_CUDA_CHECK(cudaMalloc(&ctx->d_buf, dneed + dneed / 2));
        ctx->d_cap = dneed + dneed / 2;
    }
    if (ctx->h_cap < hneed) {
        if (ctx->h_buf) cudaFreeHost(ctx->h_buf);
        ctx->h_buf = nullptr; ctx->h_cap = 0;
        HM_CUDA_CHECK(cudaMallocHost(&ctx->h_buf, hneed + hneed / 2));
        ctx->h_cap = hneed + hneed / 2;
    }
    return HM_OK;
}

static void copy_rows(uint8_t* dst, const uint8_t* src, int64_t n, int64_t stride)
{
    if (stride == HM_DESC_BYTES) {
        memcpy(dst, src, (size_t)n * HM_DESC_BYTES);
    } else {
        for (int64_t i = 0; i < n; ++i) memcpy(dst + i * HM_DESC_BYTES, src + i * stride, HM_DESC_BYTES);
    }
}

// Single-launch path for small problems (hm_small.cu): the kernel publishes its results and then the call's epoch into
// mapped pinned memory; the host polls that word instead of synchronising the stream.  `res` = host view of the result
// block [count, epoch, pad, pad][q][t][d].  Returns HM_OK once the results are visible.
static int small_match_run(hm_context* ctx, const uint8_t* q_dev, int64_t nq, const uint8_t* t_dev, int64_t nt, unsigned flags,
                           const RatioLut& lut, int thr, int* res)
{
    int* res_dev = nullptr;
    HM_CUDA_CHECK(cudaHostGetDevicePointer(reinterpret_cast<void**>(&res_dev), res, 0));
    const unsigned epoch = ++ctx->small_epoch ? ctx->small_epoch : ++ctx->small_epoch;      // never 0
    volatile int* vres = res;
    vres[1] = 0;
    int rc = launch_small_match(q_dev, nq, t_dev, nt, flags, lut, thr, res_dev, epoch, ctx->stream);
    if (rc != HM_OK) return rc;
    for (unsigned long long spins = 1;; ++spins) {
        if ((unsigned)vres[1] == epoch) break;
        if ((spins & 0x3FFF) == 0) {                  // the failure check: a kernel that died never publishes
            // after ~1 ms of polling the device is evidently busy with something else: stop burning the core
            const cudaError_t e = spins > (1ull << 20) ? cudaStreamSynchronize(ctx->stream) : cudaStreamQuery(ctx->stream);
            if (e == cudaSuccess) {
                if ((unsigned)vres[1] == epoch) break;
                set_error("small-problem kernel finished without publishing its result");
                return HM_ERR_CUDA;
            }
            if (e != cudaErrorNotReady) {
                set_error("small-problem kernel failed: %s", cudaGetErrorString(e));
                return HM_ERR_CUDA;
            }
        }
    }
    __atomic_thread_fence(__ATOMIC_ACQUIRE);
    return HM_OK;
}

// hm_small.cu is a POPC kernel: it serves AUTO and POPC calls only, so an explicit tensor-core variant runs the core
// that was asked for at every size
static bool small_path(int variant, int64_t nq, int64_t nt)
{
    return (variant == HM_VARIANT_AUTO || variant == HM_VARIANT_POPC) && small_match_eligible(nq, nt) &&
           !(g_prof_start && g_prof_stop);
}

HM_API int hm_match_host(hm_context* ctx, const uint8_t* query_host, int64_t nq, int64_t q_stride,
                         const uint8_t* train_host, int64_t nt, int64_t t_stride, unsigned flags,
                         const uint16_t* ratio_lut_host, double dist_threshold, int variant, int32_t* out_q_host,
                         int32_t* out_t_host, int32_t* out_d_host, int32_t* out_count_host)
{
    if (!ctx || nq < 0 || nt < 0 || !out_count_host || (nq > 0 && (!query_host || !out_q_host || !out_t_host || !out_d_host)) ||
        (nt > 0 && !train_host) || q_stride < HM_DESC_BYTES || t_stride < HM_DESC_BYTES) {
        set_error("hm_match_host: bad arguments");
        return HM_ERR_INVALID_ARGUMENT;
    }
    *out_count_host = 0;
    if (nq == 0 || nt == 0) return HM_OK;          // cv2: no matches when either side is empty
    const size_t qb = align_up((size_t)nq * HM_DESC_BYTES, 1024), tb = align_up((size_t)nt * HM_DESC_BYTES, 1024);
    const size_t rb = align_up((size_t)nq * 12 + 16, 1024);      // [count | pad][q][t][d]
    const size_t wsb = align_up(hm_workspace_bytes(nq, nt, 1, variant), 1024);
    int rc = ctx_reserve(ctx, qb + tb + rb + wsb, qb + tb + rb);
    if (rc != HM_OK) return rc;
    uint8_t *dq = ctx->d_buf, *dt = dq + qb, *dr = dt + tb, *dw = dr + rb;
    uint8_t *hq = ctx->h_buf, *ht = hq + qb, *hr = ht + tb;
    copy_rows(hq, query_host, nq, q_stride);
    copy_rows(ht, train_host, nt, t_stride);
    if (small_path(variant, nq, nt)) {
        // one launch, inputs read from the pinned staging buffer, results polled: no copies, no synchronisation
        RatioLut lut;
        int thr;
        if ((rc = build_filter_args(flags, ratio_lut_host, dist_threshold, &lut, &thr)) != HM_OK) return rc;
        uint8_t* hq_dev = nullptr;
        HM_CUDA_CHECK(cudaHostGetDevicePointer(reinterpret_cast<void**>(&hq_dev), hq, 0));
        if ((rc = small_match_run(ctx, hq_dev, nq, hq_dev + qb, nt, flags, lut, thr, reinterpret_cast<int*>(hr))) != HM_OK) return rc;
        const int32_t n = *reinterpret_cast<int32_t*>(hr);
        const int32_t* h_q = reinterpret_cast<int32_t*>(hr + 16);
        memcpy(out_q_host, h_q, (size_t)n * 4);
        memcpy(out_t_host, h_q + nq, (size_t)n * 4);
        memcpy(out_d_host, h_q + 2 * nq, (size_t)n * 4);
        *out_count_host = n;
        return HM_OK;
    }
    int32_t* d_count = reinterpret_cast<int32_t*>(dr);
    int32_t* d_q = reinterpret_cast<int32_t*>(dr + 16);
    int32_t* d_t = d_q + nq;
    int32_t* d_d = d_t + nq;
    GraphKey key;
    fill_key(&key, 0, nq, nt, flags, variant, 0, ratio_lut_host, dist_threshold);
    key.ptr[0] = ctx->d_buf; key.ptr[1] = ctx->h_buf;
    rc = run_cached_graph(ctx, key, [&]() -> int {
        // query and train staging are adjacent: one H2D covers both
        HM_CUDA_CHECK(cudaMemcpyAsync(dq, hq, qb + (size_t)nt * HM_DESC_BYTES, cudaMemcpyHostToDevice, ctx->stream));
        const int r = hm_match_fused(dq, nq, HM_DESC_BYTES, 0, dt, nt, HM_DESC_BYTES, 0, 1, flags, ratio_lut_host,
                                     dist_threshold, d_q, d_t, d_d, d_count, nullptr, variant, dw, wsb, ctx->stream);
        if (r != HM_OK) return r;
        HM_CUDA_CHECK(cudaMemcpyAsync(hr, dr, (size_t)nq * 12 + 16, cudaMemcpyDeviceToHost, ctx->stream));
        return HM_OK;
    });
    if (rc != HM_OK) return rc;
    HM_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    const int32_t n = *reinterpret_cast<int32_t*>(hr);
    const int32_t* h_q = reinterpret_cast<int32_t*>(hr + 16);
    memcpy(out_q_host, h_q, (size_t)n * 4);
    memcpy(out_t_host, h_q + nq, (size_t)n * 4);
    memcpy(out_d_host, h_q + 2 * nq, (size_t)n * 4);
    *out_count_host = n;
    return HM_OK;
}

// ---- resident keyframe database queried from host memory (the e2e path of the C4 workload) --------------------
// One query batch against a prepared database that stays on the device: pinned staging + H2D of the packed query,
// hm_knn2_resident (or its cross-GPU twin), D2H of the keys.  Split in two calls so that the host can do useful work
// (allocating the result objects) while the kernel runs: _begin enqueues, _end synchronises and copies out.
HM_API int hm_resident_query_begin(hm_context* ctx, const uint8_t* query_host, int64_t nq, int64_t q_stride,
                                   const void* train_prepared, int64_t nt, uint64_t train_base, int variant, int world,
                                   int rank, void* const* peer_buffers_host, int64_t max_rows, uint32_t epoch)
{
    if (!ctx || nq <= 0 || nt <= 0 || !query_host || !train_prepared || q_stride < HM_DESC_BYTES) {
        set_error("hm_resident_query_begin: bad arguments");
        return HM_ERR_INVALID_ARGUMENT;
    }
    const size_t qb = align_up((size_t)nq * HM_DESC_BYTES, 1024), kb = align_up((size_t)nq * 16, 1024);
    const size_t wsb = align_up(hm_resident_workspace_bytes(nq, nt, variant), 1024);
    int rc = ctx_reserve(ctx, qb + kb + wsb, qb + kb);
    if (rc != HM_OK) return rc;
    uint8_t *dq = ctx->d_buf, *dk = dq + qb, *dw = dk + kb;
    uint8_t *hq = ctx->h_buf, *hk = hq + qb;
    copy_rows(hq, query_host, nq, q_stride);
    HM_CUDA_CHECK(cudaMemcpyAsync(dq, hq, (size_t)nq * HM_DESC_BYTES, cudaMemcpyHostToDevice, ctx->stream));
    if (world > 1)
        rc = hm_knn2_resident_exchange(dq, nq, HM_DESC_BYTES, train_prepared, nt, train_base, world, rank, peer_buffers_host,
                                       max_rows, epoch, reinterpret_cast<uint64_t*>(dk), variant, dw, wsb, ctx->stream);
    else
        rc = hm_knn2_resident(dq, nq, HM_DESC_BYTES, train_prepared, nt, train_base, reinterpret_cast<uint64_t*>(dk), variant,
                              dw, wsb, ctx->stream);
    if (rc != HM_OK) return rc;
    HM_CUDA_CHECK(cudaMemcpyAsync(hk, dk, (size_t)nq * 16, cudaMemcpyDeviceToHost, ctx->stream));
    return HM_OK;
}

HM_API int hm_resident_query_end(hm_context* ctx, int64_t nq, uint64_t* out_keys_host)
{
    if (!ctx || nq <= 0 || !out_keys_host || !ctx->h_buf) {
        set_error("hm_resident_query_end: bad arguments");
        return HM_ERR_INVALID_ARGUMENT;
    }
    HM_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    const size_t qb = align_up((size_t)nq * HM_DESC_BYTES, 1024);
    memcpy(out_keys_host, ctx->h_buf + qb, (size_t)nq * 16);
    return HM_OK;
}

// ---- resident frames behind the context (SURVEY.md 8f ranks 1 + 2) --------------------------------------
// The reference repacks and hands BOTH frames to the matcher on every call (frontend.py:181-187,
// primitives.py:200-205).  Here a frame is uploaded once into a slot -- descriptors and, optionally, its
// keypoint positions -- and a later call matches two resident slots: per tracking step only the new frame
// crosses PCIe, and the matched point arrays of utils.py:13-19 / :41-47 come back gathered.
static inline size_t slot_points_offset(int64_t n) { return align_up((size_t)n * HM_DESC_BYTES, 256); }

HM_API int hm_frame_put(hm_context* ctx, int slot, const uint8_t* desc_host, int64_t n, int64_t stride,
                        const int32_t* points_host)
{
    if (!ctx || slot < 0 || slot >= kFrameSlots || n < 0 || (n > 0 && (!desc_host || stride < HM_DESC_BYTES))) {
        set_error("hm_frame_put: bad arguments (slots 0..%d)", kFrameSlots - 1);
        return HM_ERR_INVALID_ARGUMENT;
    }
    FrameSlot& f = ctx->slots[slot];
    // the slot advertises rows only once their copy is enqueued: a failed allocation below leaves it empty
    f.n = 0;
    f.has_points = points_host != nullptr;      // an empty frame may still be "stored with positions"
    if (n == 0) return HM_OK;
    f.has_points = false;
    const size_t bytes = slot_points_offset(n) + (size_t)n * 8;
    if (f.cap < bytes) {
        HM_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));        // kernels may still read the old buffer
        if (f.d) cudaFree(f.d);
        if (f.h) cudaFreeHost(f.h);
        f.d = f.h = nullptr; f.cap = f.h_cap = 0;
        HM_CUDA_CHECK(cudaMalloc(&f.d, bytes + bytes / 2));
        if (cudaMallocHost(&f.h, bytes + bytes / 2) != cudaSuccess) {
            cudaGetLastError();
            cudaFree(f.d);
            f.d = f.h = nullptr;
            set_error("hm_frame_put: cudaMallocHost(%zu) failed", bytes + bytes / 2);
            return HM_ERR_CUDA;
        }
        f.cap = f.h_cap = bytes + bytes / 2;
    }
    if (!f.uploaded) HM_CUDA_CHECK(cudaEventCreateWithFlags(&f.uploaded, cudaEventDisableTiming));
    else HM_CUDA_CHECK(cudaEventSynchronize(f.uploaded));          // the previous copy has left the staging buffer
    copy_rows(f.h, desc_host, n, stride);
    size_t copy_bytes = (size_t)n * HM_DESC_BYTES;
    if (points_host) {
        memcpy(f.h + slot_points_offset(n), points_host, (size_t)n * 8);
        copy_bytes = bytes;
    }
    // stream order also keeps earlier matches that read this slot ahead of the overwrite
    HM_CUDA_CHECK(cudaMemcpyAsync(f.d, f.h, copy_bytes, cudaMemcpyHostToDevice, ctx->stream));
    HM_CUDA_CHECK(cudaEventRecord(f.uploaded, ctx->stream));
    f.n = n;
    f.has_points = points_host != nullptr;
    return HM_OK;
}

// Descriptors computed on the device, straight into a frame slot (SURVEY.md 8f rank 3): the image and the keypoints
// cv2's detector found go up, the pyramid / blur / rBRIEF kernels of hm_orb.cu write the slot's descriptor rows, and
// nothing comes back unless out_desc_host asks for a copy.  Replaces the descriptor half of
// /root/reference/feature_detectors.py:25-26 (cv2.ORB.detectAndCompute) + the hm_frame_put upload.
HM_API int hm_frame_put_orb(hm_context* ctx, int slot, const uint8_t* image_host, int rows, int cols, int64_t row_stride,
                            int channels, int n_levels, const float* kp_xy_host, const float* kp_angle_deg_host,
                            const int32_t* kp_octave_host, int64_t n, const int32_t* points_host, uint8_t* out_desc_host)
{
    if (!ctx || slot < 0 || slot >= kFrameSlots || n < 0 || !image_host || (channels != 1 && channels != 3) ||
        row_stride < (int64_t)cols * channels || (n > 0 && (!kp_xy_host || !kp_angle_deg_host || !kp_octave_host))) {
        set_error("hm_frame_put_orb: bad arguments (slots 0..%d, uint8 image with 1 or 3 channels)", kFrameSlots - 1);
        return HM_ERR_INVALID_ARGUMENT;
    }
    const size_t orb_ws = orb_workspace_bytes(rows, cols, n_levels);
    if (!orb_ws) return HM_ERR_INVALID_ARGUMENT;                     // orb_geometry set the error
    for (int64_t i = 0; i < n; ++i)
        if (kp_octave_host[i] < 0 || kp_octave_host[i] >= n_levels) {
            set_error("hm_frame_put_orb: keypoint %lld has octave %d, pyramid has %d levels", (long long)i, kp_octave_host[i], n_levels);
            return HM_ERR_INVALID_ARGUMENT;
        }
    FrameSlot& f = ctx->slots[slot];
    f.n = 0;
    f.has_points = points_host != nullptr;
    if (n == 0) return HM_OK;
    f.has_points = false;
    // staging / scratch: [image | xy | cs | octave] then the pyramid workspace (device only)
    const size_t img_b = align_up((size_t)rows * cols * channels, 256), f2_b = align_up((size_t)n * 8, 256), oct_b = align_up((size_t)n * 4, 256);
    const size_t in_b = img_b + 2 * f2_b + oct_b;
    if (ctx->staged) HM_CUDA_CHECK(cudaEventSynchronize(ctx->staged));   // the previous put has left the staging buffer
    int rc = ctx_reserve(ctx, in_b + orb_ws, in_b);
    if (rc != HM_OK) return rc;
    const size_t bytes = slot_points_offset(n) + (size_t)n * 8;
    if (f.cap < bytes) {
        HM_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
        if (f.d) cudaFree(f.d);
        if (f.h) cudaFreeHost(f.h);
        f.d = f.h = nullptr; f.cap = f.h_cap = 0;
        HM_CUDA_CHECK(cudaMalloc(&f.d, bytes + bytes / 2));
        if (cudaMallocHost(&f.h, bytes + bytes / 2) != cudaSuccess) {
            cudaGetLastError();
            cudaFree(f.d);
            f.d = f.h = nullptr;
            set_error("hm_frame_put_orb: cudaMallocHost(%zu) failed", bytes + bytes / 2);
            return HM_ERR_CUDA;
        }
        f.cap = f.h_cap = bytes + bytes / 2;
    }
    if (!f.uploaded) HM_CUDA_CHECK(cudaEventCreateWithFlags(&f.uploaded, cudaEventDisableTiming));
    else HM_CUDA_CHECK(cudaEventSynchronize(f.uploaded));
    if (!ctx->staged) HM_CUDA_CHECK(cudaEventCreateWithFlags(&ctx->staged, cudaEventDisableTiming));
    uint8_t* h = ctx->h_buf;
    for (int r = 0; r < rows; ++r) memcpy(h + (size_t)r * cols * channels, image_host + (size_t)r * row_stride, (size_t)cols * channels);
    memcpy(h + img_b, kp_xy_host, (size_t)n * 8);
    orb_angles_to_cs(kp_angle_deg_host, n, reinterpret_cast<float*>(h + img_b + f2_b));
    memcpy(h + img_b + 2 * f2_b, kp_octave_host, (size_t)n * 4);
    uint8_t* d = ctx->d_buf;
    HM_CUDA_CHECK(cudaMemcpyAsync(d, h, in_b, cudaMemcpyHostToDevice, ctx->stream));
    HM_CUDA_CHECK(cudaEventRecord(ctx->staged, ctx->stream));
    if ((rc = launch_orb_pyramid(d, rows, cols, (long long)cols * channels, channels, n_levels, d + in_b, orb_ws, ctx->stream)) != HM_OK) return rc;
    if ((rc = launch_orb_describe(d + in_b, rows, cols, n_levels, reinterpret_cast<const float*>(d + img_b),
                                  reinterpret_cast<const float*>(d + img_b + f2_b), reinterpret_cast<const int*>(d + img_b + 2 * f2_b), n,
                                  f.d, HM_DESC_BYTES, ctx->stream)) != HM_OK) return rc;
    if (points_host) {
        memcpy(f.h + slot_points_offset(n), points_host, (size_t)n * 8);
        HM_CUDA_CHECK(cudaMemcpyAsync(f.d + slot_points_offset(n), f.h + slot_points_offset(n), (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
    }
    if (out_desc_host) HM_CUDA_CHECK(cudaMemcpyAsync(f.h, f.d, (size_t)n * HM_DESC_BYTES, cudaMemcpyDeviceToHost, ctx->stream));
    HM_CUDA_CHECK(cudaEventRecord(f.uploaded, ctx->stream));
    f.n = n;
    f.has_points = points_host != nullptr;
    if (out_desc_host) {
        HM_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
        memcpy(out_desc_host, f.h, (size_t)n * HM_DESC_BYTES);
    }
    return HM_OK;
}

HM_API int hm_frame_match(hm_context* ctx, int train_slot, int query_slot, unsigned flags, const uint16_t* ratio_lut_host,
                          double dist_threshold, int variant, int32_t* out_q_host, int32_t* out_t_host,
                          int32_t* out_d_host, int32_t* out_query_pts_host, int32_t* out_train_pts_host,
                          int32_t* out_count_host)
{
    if (!ctx || train_slot < 0 || train_slot >= kFrameSlots || query_slot < 0 || query_slot >= kFrameSlots ||
        !out_count_host) {
        set_error("hm_frame_match: bad arguments");
        return HM_ERR_INVALID_ARGUMENT;
    }
    const FrameSlot& T = ctx->slots[train_slot];
    const FrameSlot& Q = ctx->slots[query_slot];
    const bool want_pts = out_query_pts_host && out_train_pts_host;
    if (want_pts && (!T.has_points || !Q.has_points)) {
        set_error("hm_frame_match: matched points requested but a frame was stored without positions");
        return HM_ERR_INVALID_ARGUMENT;
    }
    *out_count_host = 0;
    const int64_t nq = Q.n, nt = T.n;
    if (nq == 0 || nt == 0) return HM_OK;              // cv2: no matches when either side is empty
    // result block: [count | pad][q][t][d][query pts][train pts], one D2H
    const size_t rb = align_up(16 + (size_t)nq * 12 + (want_pts ? (size_t)nq * 16 : 0), 1024);
    const size_t wsb = align_up(hm_workspace_bytes(nq, nt, 1, variant), 1024);
    int rc = ctx_reserve(ctx, rb + wsb, rb);
    if (rc != HM_OK) return rc;
    uint8_t *dr = ctx->d_buf, *dw = dr + rb, *hr = ctx->h_buf;
    int32_t* d_count = reinterpret_cast<int32_t*>(dr);
    int32_t* d_q = reinterpret_cast<int32_t*>(dr + 16);
    int32_t* d_t = d_q + nq;
    int32_t* d_d = d_t + nq;
    int32_t* d_pq = d_d + nq;          // 16 + 12 nq bytes: 8-byte aligned when nq is even; padded below otherwise
    if (nq & 1) ++d_pq;
    int32_t* d_pt = d_pq + 2 * nq;
    if (!want_pts && small_path(variant, nq, nt)) {
        RatioLut lut;
        int thr;
        if ((rc = build_filter_args(flags, ratio_lut_host, dist_threshold, &lut, &thr)) != HM_OK) return rc;
        if ((rc = small_match_run(ctx, Q.d, nq, T.d, nt, flags, lut, thr, reinterpret_cast<int*>(hr))) != HM_OK) return rc;
        const int32_t n = *reinterpret_cast<int32_t*>(hr);
        const int32_t* h_q = reinterpret_cast<int32_t*>(hr + 16);
        if (out_q_host) memcpy(out_q_host, h_q, (size_t)n * 4);
        if (out_t_host) memcpy(out_t_host, h_q + nq, (size_t)n * 4);
        if (out_d_host) memcpy(out_d_host, h_q + 2 * nq, (size_t)n * 4);
        *out_count_host = n;
        return HM_OK;
    }
    const size_t out_bytes = want_pts ? (size_t)(reinterpret_cast<uint8_t*>(d_pt + 2 * nq) - dr) : 16 + (size_t)nq * 12;
    GraphKey key;
    fill_key(&key, 1, nq, nt, flags, variant, want_pts ? 1 : 0, ratio_lut_host, dist_threshold);
    key.ptr[0] = ctx->d_buf; key.ptr[1] = ctx->h_buf; key.ptr[2] = Q.d; key.ptr[3] = T.d;
    rc = run_cached_graph(ctx, key, [&]() -> int {
        int r = hm_match_fused(Q.d, nq, HM_DESC_BYTES, 0, T.d, nt, HM_DESC_BYTES, 0, 1, flags, ratio_lut_host,
                               dist_threshold, d_q, d_t, d_d, d_count, nullptr, variant, dw, wsb, ctx->stream);
        if (r != HM_OK) return r;
        if (want_pts) {
            r = hm_gather_points(d_q, d_t, d_count, nq, 1, reinterpret_cast<const int32_t*>(Q.d + slot_points_offset(nq)),
                                 nq, reinterpret_cast<const int32_t*>(T.d + slot_points_offset(nt)), nt, d_pq, d_pt,
                                 ctx->stream);
            if (r != HM_OK) return r;
        }
        HM_CUDA_CHECK(cudaMemcpyAsync(hr, dr, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
        return HM_OK;
    });
    if (rc != HM_OK) return rc;
    HM_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    const int32_t n = *reinterpret_cast<int32_t*>(hr);
    const int32_t* h_q = reinterpret_cast<int32_t*>(hr + 16);
    if (out_q_host) memcpy(out_q_host, h_q, (size_t)n * 4);
    if (out_t_host) memcpy(out_t_host, h_q + nq, (size_t)n * 4);
    if (out_d_host) memcpy(out_d_host, h_q + 2 * nq, (size_t)n * 4);
    if (want_pts) {
        const int32_t* h_pq = h_q + 3 * nq + (nq & 1);
        memcpy(out_query_pts_host, h_pq, (size_t)n * 8);
        memcpy(out_train_pts_host, h_pq + 2 * nq, (size_t)n * 8);
    }
    *out_count_host = n;
    return HM_OK;
}

}  // extern "C"
