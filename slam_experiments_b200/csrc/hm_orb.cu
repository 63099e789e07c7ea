// ORB descriptor stage on the device (SURVEY.md 8f rank 3): the step in front of the matcher.
//
// Replaces the descriptor half of cv2.ORB.detectAndCompute as the reference calls it
// (/root/reference/feature_detectors.py:25-26, from /root/reference/frontend.py:245-249): given the image and the
// keypoints cv2's detector produced (position, angle, octave), build the scale pyramid, blur it, and take the 256
// steered-BRIEF comparisons per keypoint -- straight into a resident frame slot, so descriptors never visit the host.
// Keypoint DETECTION (FAST + Harris + per-level retainBest) stays with cv2 on the host; out of scope here.
//
// Bit-exactness contract = oracle/orb_oracle.py, which is pinned against cv2 4.13 (opencv-python-headless wheel):
//   gray     (B 3735 + G 19235 + R 9798 + 2^14) >> 15
//   level L  size round(rows / 1.2f^L) x round(cols / 1.2f^L) (float32, computed on the host with the same libm as cv2),
//            resized from level L-1 by the bit-exact bilinear resampler: coefficients round(frac * 256) from IEEE
//            double arithmetic without contraction, (cy0 (cx0 p00 + cx1 p01) + cy1 (cx0 p10 + cx1 p11) + 2^15) >> 16
//   frame    32 pixels of BORDER_REFLECT_101 around every level (un-blurred)
//   blur     7 x 7 sigma 2 separable FLOAT filter with cv2's summation order: fused multiply-adds in the vector body
//            of each pass, multiply-then-add in the scalar tails (x >= 32 floor(w/32) for rows, x >= 4 floor(w/4) for
//            columns), round half to even
//   rBRIEF   x' = rint(x cos - y sin), y' = rint(x sin + y cos) in float32 without contraction; bit k of byte i is
//            I(p[16 i + 2 k]) < I(p[16 i + 2 k + 1]); cos / sin come from the host (libm's double cos / sin rounded to
//            float, as in cv2)
#include <math.h>
#include <string.h>

#include "hm_common.cuh"

namespace hm {
namespace {

constexpr int kBorder = HM_ORB_BORDER;
constexpr int kMaxLevels = HM_ORB_MAX_LEVELS;

struct OrbLevel {
    int rows, cols;                  // interior size
    int stride;                      // framed row length in bytes (cols + 2 * border, padded to 16)
    long long offset;                // byte offset of the framed level inside a plane
    float inv_scale;                 // 1.f / (float)pow(1.2f, level)
    double sx, sy;                   // resize source step: 1.0 / ((double)cols / prev_cols), same for rows
};

struct OrbGeometry {
    int n_levels;
    long long plane_bytes;
    OrbLevel lv[kMaxLevels];
};

// Host arithmetic, identical to ORB_Impl::detectAndCompute's layer set-up: getScale() is (float)pow((double)1.2f, level).
// Accepted: each side of level 0 at most 16384, 1 .. 16 levels, and every level more than 32 pixels on both sides
// (checked in the loop; level 0 is the image itself).
int orb_geometry(int rows, int cols, int n_levels, OrbGeometry* g)
{
    if (rows > 16384 || cols > 16384 || n_levels < 1 || n_levels > kMaxLevels) {
        set_error("hm_orb: image %d x %d with %d levels is out of range (each side at most 16384, levels 1 .. %d)", rows, cols,
                  n_levels, kMaxLevels);
        return HM_ERR_INVALID_ARGUMENT;
    }
    memset(g, 0, sizeof(*g));
    g->n_levels = n_levels;
    long long off = 0;
    int prev_rows = rows, prev_cols = cols;
    for (int l = 0; l < n_levels; ++l) {
        OrbLevel& L = g->lv[l];
        const float scale = (float)pow((double)1.2f, (double)l);
        L.inv_scale = 1.0f / scale;
        L.rows = (int)lrintf((float)rows * L.inv_scale);
        L.cols = (int)lrintf((float)cols * L.inv_scale);
        if (L.rows <= kBorder || L.cols <= kBorder) {     // the reflected frame must fit inside the level
            set_error("hm_orb: level %d of a %d x %d image is %d x %d; every level must be more than %d pixels on both sides "
                      "(the reflected frame)", l, rows, cols, L.rows, L.cols, kBorder);
            return HM_ERR_INVALID_ARGUMENT;
        }
        L.stride = (L.cols + 2 * kBorder + 15) / 16 * 16;
        L.offset = off;
        L.sx = 1.0 / ((double)L.cols / (double)prev_cols);
        L.sy = 1.0 / ((double)L.rows / (double)prev_rows);
        off += (long long)L.stride * (L.rows + 2 * kBorder);
        off = (off + 255) / 256 * 256;
        prev_rows = L.rows; prev_cols = L.cols;
    }
    g->plane_bytes = off;
    return HM_OK;
}

__device__ __forceinline__ int reflect101(int i, int n) { return i < 0 ? -i : (i >= n ? 2 * n - 2 - i : i); }

// ---- level 0: gray conversion + frame ------------------------------------------------------------------
struct Level0Params {
    const uint8_t* image;
    long long row_stride;
    int channels;
    uint8_t* raw;
    OrbLevel L;
};

__global__ void __launch_bounds__(256) hm_orb_level0_kernel(const Level0Params P)
{
    const int X = blockIdx.x * blockDim.x + threadIdx.x, Y = blockIdx.y;
    if (X >= P.L.cols + 2 * kBorder) return;
    const int sx = reflect101(X - kBorder, P.L.cols), sy = reflect101(Y - kBorder, P.L.rows);
    const uint8_t* src = P.image + (long long)sy * P.row_stride + (long long)sx * P.channels;
    unsigned v;
    if (P.channels == 1) v = src[0];
    else v = (src[0] * 3735u + src[1] * 19235u + src[2] * 9798u + (1u << 14)) >> 15;    // cv2 BGR2GRAY, 15-bit fixed point
    P.raw[P.L.offset + (long long)Y * P.L.stride + X] = (uint8_t)v;
}

// ---- level L from level L-1: bit-exact bilinear (cv2 INTER_LINEAR_EXACT), framed ------------------------
struct ResizeParams {
    uint8_t* raw;
    OrbLevel src, dst;
};

// offset and 8.8 coefficient of one output coordinate (interpolationLinear::getCoeffs, softdouble = IEEE double)
__device__ __forceinline__ void linear_coeff(int d, double scale, int src_n, int& ofs, int& c1)
{
    const double fval = __dsub_rn(__dmul_rn(scale, (double)d + 0.5), 0.5);
    const int ival = (int)floor(fval);
    if (ival >= 0 && src_n > 1) {
        if (ival < src_n - 1) {
            ofs = ival;
            c1 = __double2int_rn(__dmul_rn(__dsub_rn(fval, (double)ival), 256.0));
        } else {
            ofs = src_n - 1; c1 = 0;
        }
    } else {
        ofs = 0; c1 = 0;
    }
}

__global__ void __launch_bounds__(256) hm_orb_resize_kernel(const ResizeParams P)
{
    const int X = blockIdx.x * blockDim.x + threadIdx.x, Y = blockIdx.y;
    if (X >= P.dst.cols + 2 * kBorder) return;
    const int dx = reflect101(X - kBorder, P.dst.cols), dy = reflect101(Y - kBorder, P.dst.rows);
    int xo, x1, yo, y1;
    linear_coeff(dx, P.dst.sx, P.src.cols, xo, x1);
    linear_coeff(dy, P.dst.sy, P.src.rows, yo, y1);
    const int xn = min(xo + 1, P.src.cols - 1), yn = min(yo + 1, P.src.rows - 1);
    const uint8_t* s = P.raw + P.src.offset + (long long)kBorder * P.src.stride + kBorder;
    const unsigned p00 = s[(long long)yo * P.src.stride + xo], p01 = s[(long long)yo * P.src.stride + xn];
    const unsigned p10 = s[(long long)yn * P.src.stride + xo], p11 = s[(long long)yn * P.src.stride + xn];
    const unsigned x0 = 256 - x1, y0 = 256 - y1;
    const unsigned h0 = x0 * p00 + x1 * p01, h1 = x0 * p10 + x1 * p11;      // 8.8
    const unsigned v = (y0 * h0 + y1 * h1 + (1u << 15)) >> 16;              // 16.16, round to nearest
    P.raw[P.dst.offset + (long long)Y * P.dst.stride + X] = (uint8_t)v;
}

// ---- blur: every level in one launch --------------------------------------------------------------------
struct BlurParams {
    const uint8_t* raw;
    uint8_t* blurred;
    OrbGeometry G;
};

// cv2.getGaussianKernel(7, 2, CV_32F): bit patterns
__constant__ unsigned kGauss7[7] = {0x3d8fafb1u, 0x3e06387eu, 0x3e434a39u, 0x3e5d4ae0u, 0x3e434a39u, 0x3e06387eu, 0x3d8fafb1u};

__global__ void __launch_bounds__(256) hm_orb_blur_kernel(const BlurParams P)
{
    const OrbLevel& L = P.G.lv[blockIdx.z];
    const int X = blockIdx.x * blockDim.x + threadIdx.x, Y = blockIdx.y;
    if (X >= L.cols + 2 * kBorder || Y >= L.rows + 2 * kBorder) return;
    const long long at = L.offset + (long long)Y * L.stride + X;
    const int x = X - kBorder, y = Y - kBorder;
    if (x < 0 || y < 0 || x >= L.cols || y >= L.rows) {          // the frame keeps its un-blurred values
        P.blurred[at] = P.raw[at];
        return;
    }
    float g[7];
#pragma unroll
    for (int k = 0; k < 7; ++k) g[k] = __uint_as_float(kGauss7[k]);
    const bool row_fused = x < (L.cols / 32) * 32, col_fused = x < (L.cols / 4) * 4;
    float r[7];
#pragma unroll
    for (int j = 0; j < 7; ++j) {
        const uint8_t* p = P.raw + at + (long long)(j - 3) * L.stride - 3;
        float s = __fmul_rn(g[0], (float)p[0]);
#pragma unroll
        for (int k = 1; k < 7; ++k)
            s = row_fused ? __fmaf_rn(g[k], (float)p[k], s) : __fadd_rn(s, __fmul_rn(g[k], (float)p[k]));
        r[j] = s;
    }
    float c = __fmul_rn(g[3], r[3]);
#pragma unroll
    for (int k = 1; k < 4; ++k) {
        const float pair = __fadd_rn(r[3 + k], r[3 - k]);
        c = col_fused ? __fmaf_rn(g[3 + k], pair, c) : __fadd_rn(c, __fmul_rn(g[3 + k], pair));
    }
    P.blurred[at] = (uint8_t)min(max(__float2int_rn(c), 0), 255);
}

// ---- rBRIEF: one warp per keypoint, lane = descriptor byte ------------------------------------------------
struct DescribeParams {
    const uint8_t* blurred;
    OrbGeometry G;
    const float2* xy;                // level-0 pixel coordinates (KeyPoint.pt)
    const float2* cs;                // (cos, sin) of the keypoint angle
    const int* octave;
    long long n;
    uint8_t* out;
    long long out_stride;
};

__constant__ signed char kPattern31[512][2] = {
#include "hm_orb_pattern.inc"
};

constexpr int kDescribeWarps = 8;

__global__ void __launch_bounds__(kDescribeWarps * 32) hm_orb_describe_kernel(const DescribeParams P)
{
    __shared__ float2 pat[512];
    for (int i = threadIdx.x; i < 512; i += blockDim.x) pat[i] = make_float2((float)kPattern31[i][0], (float)kPattern31[i][1]);
    __syncthreads();
    const long long j = (long long)blockIdx.x * kDescribeWarps + (threadIdx.x >> 5);
    if (j >= P.n) return;
    const int lane = threadIdx.x & 31;
    const int lv = min(max(P.octave[j], 0), P.G.n_levels - 1);
    const OrbLevel& L = P.G.lv[lv];
    const float2 pt = P.xy[j], cs = P.cs[j];
    const int W = L.cols + 2 * kBorder, H = L.rows + 2 * kBorder;
    const int cx = __float2int_rn(__fmul_rn(pt.x, L.inv_scale)) + kBorder;
    const int cy = __float2int_rn(__fmul_rn(pt.y, L.inv_scale)) + kBorder;
    const uint8_t* plane = P.blurred + L.offset;
    unsigned byte = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        int v[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const float2 p = pat[lane * 16 + 2 * k + e];
            const int ix = __float2int_rn(__fsub_rn(__fmul_rn(p.x, cs.x), __fmul_rn(p.y, cs.y)));
            const int iy = __float2int_rn(__fadd_rn(__fmul_rn(p.x, cs.y), __fmul_rn(p.y, cs.x)));
            // keypoints from cv2's detector stay 31 pixels inside their level, so the 32-pixel frame covers every
            // sample; the clamp only keeps hand-made keypoints memory-safe (cv2 reads out of bounds there)
            const int X = min(max(cx + ix, 0), W - 1), Y = min(max(cy + iy, 0), H - 1);
            v[e] = plane[(long long)Y * L.stride + X];
        }
        byte |= (unsigned)(v[0] < v[1]) << k;
    }
    P.out[j * P.out_stride + lane] = (uint8_t)byte;
}

}  // namespace

// ---- launch sequences (used by the C entry points below and by the context in hm_api.cu) -----------------
size_t orb_workspace_bytes(int rows, int cols, int n_levels)
{
    OrbGeometry g;
    if (orb_geometry(rows, cols, n_levels, &g) != HM_OK) return 0;
    return 256 + 2 * (size_t)g.plane_bytes;
}

int launch_orb_pyramid(const uint8_t* image, int rows, int cols, long long row_stride, int channels, int n_levels, void* ws,
                       size_t ws_bytes, cudaStream_t stream)
{
    OrbGeometry g;
    int rc = orb_geometry(rows, cols, n_levels, &g);
    if (rc != HM_OK) return rc;
    if (!image || (channels != 1 && channels != 3) || row_stride < (long long)cols * channels) {
        set_error("hm_orb_build_pyramid: image must be non-null uint8 with 1 (gray) or 3 (BGR) channels");
        return HM_ERR_INVALID_ARGUMENT;
    }
    const size_t need = 256 + 2 * (size_t)g.plane_bytes;
    if (!ws || ws_bytes < need) {
        set_error("workspace too small: need %zu bytes, got %zu", need, ws_bytes);
        return HM_ERR_WORKSPACE;
    }
    uint8_t* raw = static_cast<uint8_t*>(ws) + 256;
    uint8_t* blurred = raw + g.plane_bytes;
    {
        Level0Params P{image, row_stride, channels, raw, g.lv[0]};
        dim3 grid((unsigned)ceil_div(g.lv[0].cols + 2 * kBorder, 256), (unsigned)(g.lv[0].rows + 2 * kBorder));
        hm_orb_level0_kernel<<<grid, 256, 0, stream>>>(P);
    }
    for (int l = 1; l < n_levels; ++l) {        // each level is resized from the previous one
        ResizeParams P{raw, g.lv[l - 1], g.lv[l]};
        dim3 grid((unsigned)ceil_div(g.lv[l].cols + 2 * kBorder, 256), (unsigned)(g.lv[l].rows + 2 * kBorder));
        hm_orb_resize_kernel<<<grid, 256, 0, stream>>>(P);
    }
    {
        BlurParams P{raw, blurred, g};
        dim3 grid((unsigned)ceil_div(g.lv[0].cols + 2 * kBorder, 256), (unsigned)(g.lv[0].rows + 2 * kBorder), (unsigned)n_levels);
        hm_orb_blur_kernel<<<grid, 256, 0, stream>>>(P);
    }
    HM_CUDA_CHECK(cudaGetLastError());
    return HM_OK;
}

int launch_orb_describe(const void* ws, int rows, int cols, int n_levels, const float* xy, const float* cs, const int* octave,
                        long long n, uint8_t* out, long long out_stride, cudaStream_t stream)
{
    OrbGeometry g;
    int rc = orb_geometry(rows, cols, n_levels, &g);
    if (rc != HM_OK) return rc;
    if (n < 0 || (n > 0 && (!ws || !xy || !cs || !octave || !out || out_stride < HM_DESC_BYTES)) ||
        ((reinterpret_cast<uintptr_t>(xy) | reinterpret_cast<uintptr_t>(cs)) & 7)) {
        set_error("hm_orb_describe: bad arguments");
        return HM_ERR_INVALID_ARGUMENT;
    }
    if (n == 0) return HM_OK;
    DescribeParams P{};
    P.blurred = static_cast<const uint8_t*>(ws) + 256 + g.plane_bytes;
    P.G = g;
    P.xy = reinterpret_cast<const float2*>(xy);
    P.cs = reinterpret_cast<const float2*>(cs);
    P.octave = octave; P.n = n; P.out = out; P.out_stride = out_stride;
    hm_orb_describe_kernel<<<(unsigned)ceil_div(n, kDescribeWarps), kDescribeWarps * 32, 0, stream>>>(P);
    HM_CUDA_CHECK(cudaGetLastError());
    return HM_OK;
}

// (cos, sin) exactly as computeOrbDescriptors takes them: angle *= (float)(CV_PI / 180.f); a = (float)cos(angle) with
// the DOUBLE cos / sin of libm on the float angle (probed: cv2 agrees with this and not with cosf / sinf on the angles
// where the two differ, tests/test_orb.py)
void orb_angles_to_cs(const float* angle_deg, long long n, float* cs)
{
    const float k = (float)(3.1415926535897932384626433832795 / 180.f);
    for (long long i = 0; i < n; ++i) {
        const float a = angle_deg[i] * k;
        cs[2 * i] = (float)cos((double)a);
        cs[2 * i + 1] = (float)sin((double)a);
    }
}

int orb_level_geometry(int rows, int cols, int level, int* out_rows, int* out_cols, float* out_inv_scale)
{
    OrbGeometry g;
    if (level < 0 || level >= kMaxLevels) {
        set_error("hm_orb_level_geometry: level out of range");
        return HM_ERR_INVALID_ARGUMENT;
    }
    const int rc = orb_geometry(rows, cols, level + 1, &g);
    if (rc != HM_OK) return rc;
    if (out_rows) *out_rows = g.lv[level].rows;
    if (out_cols) *out_cols = g.lv[level].cols;
    if (out_inv_scale) *out_inv_scale = g.lv[level].inv_scale;
    return HM_OK;
}

}  // namespace hm

using namespace hm;

extern "C" {

HM_API size_t hm_orb_workspace_bytes(int rows, int cols, int n_levels) { return orb_workspace_bytes(rows, cols, n_levels); }

HM_API int hm_orb_level_geometry(int rows, int cols, int level, int* out_rows, int* out_cols, float* out_inv_scale)
{
    return orb_level_geometry(rows, cols, level, out_rows, out_cols, out_inv_scale);
}

HM_API int hm_orb_angles_to_cs(const float* angle_deg_host, int64_t n, float* cs_host)
{
    if (n < 0 || (n > 0 && (!angle_deg_host || !cs_host))) {
        set_error("hm_orb_angles_to_cs: bad arguments");
        return HM_ERR_INVALID_ARGUMENT;
    }
    orb_angles_to_cs(angle_deg_host, n, cs_host);
    return HM_OK;
}

HM_API int hm_orb_build_pyramid(const uint8_t* image, int rows, int cols, int64_t row_stride, int channels, int n_levels,
                                void* workspace, size_t workspace_bytes, void* stream)
{
    DeviceInfo di;
    const int rc = device_info(&di);
    if (rc != HM_OK) return rc;
    return launch_orb_pyramid(image, rows, cols, row_stride, channels, n_levels, workspace, workspace_bytes,
                              static_cast<cudaStream_t>(stream));
}

HM_API int hm_orb_describe(const void* workspace, int rows, int cols, int n_levels, const float* kp_xy, const float* kp_cs,
                           const int32_t* kp_octave, int64_t n, uint8_t* out_desc, int64_t out_stride, void* stream)
{
    DeviceInfo di;
    const int rc = device_info(&di);
    if (rc != HM_OK) return rc;
    return launch_orb_describe(workspace, rows, cols, n_levels, kp_xy, kp_cs, kp_octave, n, out_desc, out_stride,
                               static_cast<cudaStream_t>(stream));
}

}  // extern "C"
