// K8 — HoVer-Net post-process (tiseg/models/segmentors/hovernet.py:283-365, hover_post_proc(fore_map, hv_map, fx,
// scale_factor)).  fx enters as two integers: the Sobel ksize = int(20 * fx + 1), odd in 1..31 (21 at fx = 1), and the
// marker obj_size = ceil(10 * fx^2) (10 at fx = 1); scale_factor is 1 or 2.
//
// The float chain (cv2.normalize -> cv2.Sobel ksize k CV_64F -> cv2.normalize -> max -> thresholds ->
// cv2.GaussianBlur 3x3) feeds two thresholds (>= 0.5, >= 0.4) and a watershed on the blurred map, so a 1-ulp
// difference can flip an integer output.  The kernels therefore reproduce OpenCV's arithmetic ORDER, not just
// its formulas (SURVEY.md Appendix A.2, re-derived in tests/cv_recipes.py and checked against cv2 bit for bit):
//   normalize (-> CV_32F): a = (float)(1/(max-min)); b = 0.f - (float)(min * a); dst = (float)fma(x, a, b) in fp64
//   Sobel k:  integer kernels of cv2.getDerivKernels; row pass = sequential taps in fp64; column pass = centre tap,
//             then k[r+t] * (R[+t] +/- R[-t]), t = 1..r, multiply and add rounded separately (no FMA);
//             BORDER_REFLECT_101, reflected again while outside (images smaller than the radius r)
//   GaussianBlur 3x3 on fp64: row pass (a/4 + b/2) + c/4, column pass b/2 + (a + c)/4
// (--fmad=false for the whole library; fma() is written out where OpenCV contracts.)
// The foreground and HV maps may be fp32, fp16 or bf16 (TI): the kernels that read them convert at the load, so the chain
// sees the fp32 values of the inputs either way.
#include <cfloat>

#include "ccl.cuh"
#include "morph.cuh"
#include "watershed.cuh"

namespace tiseg {

// cv2.getDerivKernels, indexed by tap radius r: smoothing = binomial row 2r; derivative (r >= 1) = binomial row 2r-1
// convolved with [-1, 1].  ksize k uses radius k / 2 for both passes, except ksize 1: derivative [-1, 0, 1] (radius 1),
// smoothing [1] (radius 0).  The largest coefficient, C(30, 15), is below 2^28, so every row product of an fp32 source
// is exact in fp64.
constexpr int SOBEL_RMAX = 15;                                  // ksize 31, the largest cv2.Sobel accepts
struct SobelTaps {
    double smooth[SOBEL_RMAX + 1][2 * SOBEL_RMAX + 1];
    double deriv[SOBEL_RMAX + 1][2 * SOBEL_RMAX + 1];
};
constexpr SobelTaps make_sobel_taps() {
    SobelTaps k{};
    for (int r = 0; r <= SOBEL_RMAX; ++r) {
        long long b[2 * SOBEL_RMAX + 1] = {1};                 // binomial row, built up to 2r
        for (int n = 1; n <= 2 * r; ++n) {
            if (n == 2 * r) {
                for (int i = 0; i <= 2 * r; ++i) k.deriv[r][i] = (double)((i > 0 ? b[i - 1] : 0) - (i < n ? b[i] : 0));
            }
            for (int i = n; i > 0; --i) b[i] += b[i - 1];
        }
        for (int i = 0; i <= 2 * r; ++i) k.smooth[r][i] = (double)b[i];
    }
    return k;
}
__constant__ SobelTaps c_sobel = make_sobel_taps();

__device__ __forceinline__ long long dkey(double d) {       // monotone double -> int64 (for atomicMax / atomicMin)
    long long b = __double_as_longlong(d);
    return b >= 0 ? b : b ^ 0x7fffffffffffffffll;
}
__device__ __forceinline__ double dkey_inv(long long k) { return __longlong_as_double(k >= 0 ? k : k ^ 0x7fffffffffffffffll); }

__device__ __forceinline__ void warp_minmax_commit(double lo, double hi, bool any, long long* mm) {
    long long klo = any ? dkey(lo) : 0x7fffffffffffffffll, khi = any ? dkey(hi) : (long long)0x8000000000000000ull;
    for (int s = 16; s; s >>= 1) {
        long long a = __shfl_xor_sync(0xffffffffu, klo, s), b = __shfl_xor_sync(0xffffffffu, khi, s);
        klo = a < klo ? a : klo;
        khi = b > khi ? b : khi;
    }
    if ((threadIdx.x & 31) == 0) {
        if (klo < mm[0]) atomicMin(&mm[0], klo);
        if (khi > mm[1]) atomicMax(&mm[1], khi);
    }
}

__global__ void k_mm_init(long long* mm, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { mm[2 * i] = 0x7fffffffffffffffll; mm[2 * i + 1] = (long long)0x8000000000000000ull; }
}

// min / max of the two HWC channels of the HV map (eight pixels per thread before the warp reduction)
template <class TI>
__global__ void __launch_bounds__(TISEG_THREADS)
k_hv_minmax(Geom g, const typename Pair<TI>::type* __restrict__ hv, long long* mm /* [N, 2 channels, 2] */) {
    const int n = blockIdx.y;
    const typename Pair<TI>::type* t = hv + (long long)n * g.P;
    float lx = INFINITY, hx = -INFINITY, ly = INFINITY, hy = -INFINITY;
    bool any = false;
    const long long i0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x);
    const long long stride = (long long)gridDim.x * blockDim.x;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const long long i = i0 + k * stride;
        if (i < g.P) {
            const float2 v = to_f32(t[i]);
            lx = fminf(lx, v.x); hx = fmaxf(hx, v.x); ly = fminf(ly, v.y); hy = fmaxf(hy, v.y);
            any = true;
        }
    }
    warp_minmax_commit(lx, hx, any, mm + (long long)n * 4);
    warp_minmax_commit(ly, hy, any, mm + (long long)n * 4 + 2);
}

struct NormCoef { double a, b; };
__device__ __forceinline__ NormCoef norm_coef(const long long* mm) {
    double mn = dkey_inv(mm[0]), mx = dkey_inv(mm[1]);
    double scale = (mx - mn > DBL_EPSILON) ? 1.0 / (mx - mn) : 0.0;
    float a = (float)scale;                                    // cv::normalize, rtype == CV_32F
    float b = 0.f - (float)(mn * (double)a);
    NormCoef c; c.a = (double)a; c.b = (double)b;
    return c;
}

template <class TI>
__global__ void __launch_bounds__(TISEG_THREADS)
k_hv_normalize(Geom g, const typename Pair<TI>::type* __restrict__ hv, const long long* __restrict__ mm, float* __restrict__ hdir,
               float* __restrict__ vdir) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    NormCoef ch = norm_coef(mm + (long long)px.n * 4), cv = norm_coef(mm + (long long)px.n * 4 + 2);
    float2 v = to_f32(hv[px.base + px.idx]);
    hdir[px.base + px.idx] = (float)fma((double)v.x, ch.a, ch.b);
    vdir[px.base + px.idx] = (float)fma((double)v.y, cv.a, cv.b);
}

__device__ __forceinline__ int reflect101(int i, int n) {
    if (n == 1) return 0;
    while (i < 0 || i >= n) i = i < 0 ? -i : 2 * n - 2 - i;
    return i;
}

// row pass: fp32 source -> fp64, 2R+1 sequential taps along x.  One thread = four adjacent outputs: the 2R+4 source
// values they share are read once (reflected only at the image sides); every output keeps OpenCV's tap order.
template <bool DERIV, int R>
__global__ void __launch_bounds__(TISEG_THREADS)
k_sobel_row(Geom g, const float* __restrict__ src, double* __restrict__ out) {
    constexpr int NV = 2 * R + 4;
    const int W4 = (g.W + 3) >> 2;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)W4 * g.H) return;
    const int y = (int)(t / W4), x = (int)(t - (long long)y * W4) * 4, n = blockIdx.y;
    const float* row = src + (long long)n * g.P + (long long)y * g.W;
    double* orow = out + (long long)n * g.P + (long long)y * g.W;
    const double* k = DERIV ? c_sobel.deriv[R] : c_sobel.smooth[R];
    double v[NV];
    if (x >= R && x + 3 + R < g.W) {
#pragma unroll
        for (int j = 0; j < NV; ++j) v[j] = (double)row[x - R + j];
    } else {
#pragma unroll
        for (int j = 0; j < NV; ++j) v[j] = (double)row[reflect101(x - R + j, g.W)];
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        if (x + q >= g.W) break;
        double s = k[0] * v[q];
#pragma unroll
        for (int tt = 1; tt <= 2 * R; ++tt) s = s + k[tt] * v[q + tt];
        orow[x + q] = s;
    }
}

// column pass (symmetric pairing, separate multiply and add) + min / max of the result.  One thread = four
// vertically adjacent outputs of one column (2R+4 row values read once, each read coalesced over the warp).
// The bound of one block per SM lets ptxas give the pass the registers it needs: with the plain bound it stopped at an
// occupancy step (48, 64 or 80 registers) and spilled 8-32 bytes at radii 4 and 7-11.
template <bool DERIV, int R>
__global__ void __launch_bounds__(TISEG_THREADS, 1)
k_sobel_col(Geom g, const double* __restrict__ rowbuf, double* __restrict__ out, long long* mm /* [N, 2] */) {
    constexpr int NV = 2 * R + 4;
    const int H4 = (g.H + 3) >> 2;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = t < (long long)H4 * g.W;
    const int n = blockIdx.y;
    double lo = 0.0, hi = 0.0;
    if (live) {
        const int y = (int)(t / g.W) * 4, x = (int)(t - (long long)(y >> 2) * g.W);
        const double* col = rowbuf + (long long)n * g.P + x;
        const double* k = DERIV ? c_sobel.deriv[R] : c_sobel.smooth[R];
        double v[NV];
        if (y >= R && y + 3 + R < g.H) {
#pragma unroll
            for (int j = 0; j < NV; ++j) v[j] = col[(long long)(y - R + j) * g.W];
        } else {
#pragma unroll
            for (int j = 0; j < NV; ++j) v[j] = col[(long long)reflect101(y - R + j, g.H) * g.W];
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            if (y + q >= g.H) break;
            double acc = DERIV ? 0.0 : __dmul_rn(k[R], v[q + R]);
#pragma unroll
            for (int d = 1; d <= R; ++d) {
                const double pair = DERIV ? __dsub_rn(v[q + R + d], v[q + R - d]) : __dadd_rn(v[q + R + d], v[q + R - d]);
                acc = __dadd_rn(acc, __dmul_rn(k[R + d], pair));
            }
            out[(long long)n * g.P + (long long)(y + q) * g.W + x] = acc;
            lo = q == 0 ? acc : fmin(lo, acc);
            hi = q == 0 ? acc : fmax(hi, acc);
        }
    }
    warp_minmax_commit(lo, hi, live, mm + (long long)n * 2);
}

// Host dispatch of one pass on its tap radius r: a chain of instantiations from the smallest radius (1 for a derivative
// pass, 0 for a smoothing pass) to SOBEL_RMAX.  Timing names "k_sobel_row<DERIV, R>" / "k_sobel_col<DERIV, R>".
inline std::string sobel_name(const char* pass, bool deriv, int r) {
    return std::string(pass) + (deriv ? "<true, " : "<false, ") + std::to_string(r) + ">";
}
inline int sobel_bad_radius(int r) {
    set_error("hover Sobel: no kernel of tap radius " + std::to_string(r));
    return TISEG_ERR_ARG;
}
template <bool DERIV, int R = (DERIV ? 1 : 0)>
int sobel_row(tiseg_ctx* c, int r, const Geom& g, dim3 grid, const float* src, double* out) {
    if (r != R) {
        if constexpr (R < SOBEL_RMAX) return sobel_row<DERIV, R + 1>(c, r, g, grid, src, out);
        else return sobel_bad_radius(r);
    }
    static const std::string name = sobel_name("k_sobel_row", DERIV, R);
    TISEG_LAUNCH_AS(c, name.c_str(), (k_sobel_row<DERIV, R>), grid, TISEG_THREADS, 0, g, src, out);
    return TISEG_OK;
}
template <bool DERIV, int R = (DERIV ? 1 : 0)>
int sobel_col(tiseg_ctx* c, int r, const Geom& g, dim3 grid, const double* rowbuf, double* out, long long* mm) {
    if (r != R) {
        if constexpr (R < SOBEL_RMAX) return sobel_col<DERIV, R + 1>(c, r, g, grid, rowbuf, out, mm);
        else return sobel_bad_radius(r);
    }
    static const std::string name = sobel_name("k_sobel_col", DERIV, R);
    TISEG_LAUNCH_AS(c, name.c_str(), (k_sobel_col<DERIV, R>), grid, TISEG_THREADS, 0, g, rowbuf, out, mm);
    return TISEG_OK;
}

template <class TI>
__global__ void k_threshold_ge(Geom g, const TI* __restrict__ x, float thr, uint8_t* __restrict__ out) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    out[px.base + px.idx] = to_f32(x[px.base + px.idx]) >= thr;
}

// hovernet.py:343-353: overall, dist (before the blur) and the raw marker mask
__global__ void __launch_bounds__(TISEG_THREADS)
k_hover_energy(Geom g, const double* __restrict__ sobh, const double* __restrict__ sobv, const long long* __restrict__ mmh,
               const long long* __restrict__ mmv, const uint8_t* __restrict__ blb, double* __restrict__ dist,
               uint8_t* __restrict__ marker) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    long long i = px.base + px.idx;
    NormCoef ch = norm_coef(mmh + (long long)px.n * 2), cv = norm_coef(mmv + (long long)px.n * 2);
    float sh = 1.f - (float)fma(sobh[i], ch.a, ch.b);
    float sv = 1.f - (float)fma(sobv[i], cv.a, cv.b);
    float ov32 = fmaxf(sh, sv);                                 // np.maximum on fp32
    int b = blb[i];
    double ov = (double)ov32 - (double)(1 - b);                 // fp32 - int32 -> fp64
    if (ov < 0.0) ov = 0.0;
    dist[i] = (1.0 - ov) * (double)b;
    int m = b - (ov >= 0.4 ? 1 : 0);
    marker[i] = m > 0;
}

__global__ void __launch_bounds__(TISEG_THREADS)
k_gauss3_row(Geom g, const double* __restrict__ src, double* __restrict__ out) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    const double* row = src + px.base + (long long)px.y * g.W;
    double a = row[reflect101(px.x - 1, g.W)], b = row[px.x], c = row[reflect101(px.x + 1, g.W)];
    out[px.base + px.idx] = __dadd_rn(__dadd_rn(0.25 * a, 0.5 * b), 0.25 * c);
}
// column pass, negated: dist = -GaussianBlur(...)
__global__ void __launch_bounds__(TISEG_THREADS)
k_gauss3_col_neg(Geom g, const double* __restrict__ src, double* __restrict__ out) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    const double* t = src + px.base + px.x;
    double a = t[(long long)reflect101(px.y - 1, g.H) * g.W], b = t[(long long)px.y * g.W],
           c = t[(long long)reflect101(px.y + 1, g.H) * g.W];
    out[px.base + px.idx] = -__dadd_rn(0.5 * b, 0.25 * __dadd_rn(a, c));
}

// cv2.morphologyEx(MORPH_OPEN, getStructuringElement(MORPH_ELLIPSE, (5, 5))): rows 00100 / 11111 x3 / 00100.
// Erosion sees the outside of the image as foreground, dilation as background (morphologyDefaultBorderValue).
template <bool ERODE>
__global__ void __launch_bounds__(TISEG_THREADS)
k_ellipse5(Geom g, const uint8_t* __restrict__ src, uint8_t* __restrict__ out, bool vec) {
    // one thread = four adjacent pixels; every row of the 5x5 ellipse (00100 / 11111 / 11111 / 11111 / 00100) is read as
    // one 32-bit word plus the two bytes on each side.  Outside the image counts as set for the erosion, clear for the
    // dilation (cv::morphologyEx default border).
    const int W4 = (g.W + 3) >> 2;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)W4 * g.H) return;
    const int y = (int)(t / W4), x = (int)(t - (long long)y * W4) * 4, n = blockIdx.y;
    const uint8_t* tile = src + (long long)n * g.P;
    const unsigned OOB = ERODE ? 1u : 0u;
    bool r[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) r[k] = ERODE;
#pragma unroll
    for (int dy = -2; dy <= 2; ++dy) {
        const int yy = y + dy;
        const bool oky = yy >= 0 && yy < g.H;
        const uint8_t* row = tile + (long long)yy * g.W;
        unsigned b[8];                                           // columns x-2 .. x+5
        if (oky && vec) {
            const unsigned w = *reinterpret_cast<const unsigned*>(row + x);
#pragma unroll
            for (int k = 0; k < 4; ++k) b[2 + k] = ((w >> (8 * k)) & 255u) != 0;
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k) b[2 + k] = (oky && x + k < g.W) ? (unsigned)(row[x + k] != 0) : OOB;
        }
        if (dy == -2 || dy == 2) {
#pragma unroll
            for (int k = 0; k < 4; ++k) r[k] = ERODE ? (r[k] && b[2 + k]) : (r[k] || b[2 + k]);
            continue;
        }
        b[0] = (oky && x - 2 >= 0) ? (unsigned)(row[x - 2] != 0) : OOB;
        b[1] = (oky && x - 1 >= 0) ? (unsigned)(row[x - 1] != 0) : OOB;
        b[6] = (oky && x + 4 < g.W) ? (unsigned)(row[x + 4] != 0) : OOB;
        b[7] = (oky && x + 5 < g.W) ? (unsigned)(row[x + 5] != 0) : OOB;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const bool all5 = b[k] && b[k + 1] && b[k + 2] && b[k + 3] && b[k + 4];
            const bool any5 = b[k] || b[k + 1] || b[k + 2] || b[k + 3] || b[k + 4];
            r[k] = ERODE ? (r[k] && all5) : (r[k] || any5);
        }
    }
    uint8_t* o = out + (long long)n * g.P + (long long)y * g.W + x;
    if (vec) *reinterpret_cast<unsigned*>(o) = (unsigned)r[0] | ((unsigned)r[1] << 8) | ((unsigned)r[2] << 16) | ((unsigned)r[3] << 24);
    else {
#pragma unroll
        for (int k = 0; k < 4; ++k) if (x + k < g.W) o[k] = r[k];
    }
}

// fore [N,H,W] and hv [N,H,W,2] of element type TI; ksize odd in 1..31
template <class TI>
int postproc_hover_dev(tiseg_ctx* c, const Geom& g, const TI* fore, const TI* hv, int ksize, int obj_size, int32_t* inst,
                       uint8_t* blb_out, double* dist_out, int32_t* marker_out) {
    int N = g.N;
    size_t total = (size_t)N * g.P;
    uint8_t* m0 = ws<uint8_t>(c, total);
    uint8_t* blb = blb_out ? blb_out : ws<uint8_t>(c, total);
    float* hdir = ws<float>(c, total); float* vdir = ws<float>(c, total);
    double* rowb = ws<double>(c, total);
    double* sobh = ws<double>(c, total); double* sobv = ws<double>(c, total);
    double* dist = dist_out ? dist_out : ws<double>(c, total);
    double* dpre = ws<double>(c, total);
    uint8_t* mk0 = ws<uint8_t>(c, total); uint8_t* mk1 = ws<uint8_t>(c, total);
    int32_t* lab = ws<int32_t>(c, total);
    int32_t* markers = marker_out ? marker_out : ws<int32_t>(c, total);
    long long* mm = ws<long long>(c, (size_t)N * 8);           // hv: [N,2,2]; sobel h: [N,2]; sobel v: [N,2]
    int* par = ws<int>(c, total); int* rank = ws<int>(c, total);
    if (!m0 || !blb || !hdir || !vdir || !rowb || !sobh || !sobv || !dist || !dpre || !mk0 || !mk1 || !lab || !markers || !mm || !par || !rank)
        return TISEG_ERR_CUDA;
    long long* mm_hv = mm; long long* mm_sh = mm + (size_t)N * 4; long long* mm_sv = mm + (size_t)N * 6;
    const typename Pair<TI>::type* hv2 = (const typename Pair<TI>::type*)hv;

    // blb = (fore >= 0.5) -> 4-connected components -> drop < 10 px (hovernet.py:294-298)
    TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "k_threshold_ge"), k_threshold_ge<TI>, warp_grid(g), TISEG_THREADS, 0, g, fore, 0.5f, m0);
    TISEG_TRY(remove_small_mask(c, g, m0, 10, 1, blb));
    // normalised H / V maps
    TISEG_LAUNCH(c, k_mm_init, (4 * N + 255) / 256, 256, 0, mm, 4 * N);
    TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "k_hv_minmax"), k_hv_minmax<TI>, dim3((unsigned)((g.P + 8 * TISEG_THREADS - 1) / (8 * TISEG_THREADS)), (unsigned)N),
                    TISEG_THREADS, 0, g, hv2, mm_hv);
    TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "k_hv_normalize"), k_hv_normalize<TI>, warp_grid(g), TISEG_THREADS, 0, g, hv2, mm_hv, hdir, vdir);
    // Sobel(h_dir, dx=1): derivative along x, smoothing along y;  Sobel(v_dir, dy=1): the transpose.  Tap radii of
    // the two kernels of cv2.getDerivKernels(ksize): ksize / 2, except ksize 1 = derivative [-1, 0, 1] and smoothing [1].
    const int rd = ksize == 1 ? 1 : ksize / 2, rs = ksize / 2;
    const dim3 rg((unsigned)(((long long)((g.W + 3) / 4) * g.H + TISEG_THREADS - 1) / TISEG_THREADS), (unsigned)N);
    const dim3 cg((unsigned)(((long long)((g.H + 3) / 4) * g.W + TISEG_THREADS - 1) / TISEG_THREADS), (unsigned)N);
    TISEG_TRY(sobel_row<true>(c, rd, g, rg, hdir, rowb));
    TISEG_TRY(sobel_col<false>(c, rs, g, cg, rowb, sobh, mm_sh));
    TISEG_TRY(sobel_row<false>(c, rs, g, rg, vdir, rowb));
    TISEG_TRY(sobel_col<true>(c, rd, g, cg, rowb, sobv, mm_sv));
    // energy, thresholds, blurred distance
    TISEG_LAUNCH(c, k_hover_energy, warp_grid(g), TISEG_THREADS, 0, g, sobh, sobv, mm_sh, mm_sv, blb, dpre, mk0);
    TISEG_LAUNCH(c, k_gauss3_row, warp_grid(g), TISEG_THREADS, 0, g, dpre, rowb);
    TISEG_LAUNCH(c, k_gauss3_col_neg, warp_grid(g), TISEG_THREADS, 0, g, rowb, dist);
    // markers: fill holes -> 5x5 elliptical opening -> 4-connected labels -> drop < obj_size (ids kept)
    TISEG_TRY(ccl_build(c, g, ImgNotMaskU8{mk0}, 1, par));
    TISEG_TRY(fill_from_complement_forest(c, g, par, mk1));
    const bool ev = (g.W % 4 == 0) && ((((uintptr_t)mk0) | ((uintptr_t)mk1)) & 3) == 0;
    TISEG_LAUNCH(c, k_ellipse5<true>, rg, TISEG_THREADS, 0, g, mk1, mk0, ev);
    TISEG_LAUNCH(c, k_ellipse5<false>, rg, TISEG_THREADS, 0, g, mk0, mk1, ev);
    TISEG_TRY(ccl_label(c, g, ImgMaskU8{mk1}, 1, lab, nullptr));
    TISEG_TRY(remove_small_labels(c, g, lab, obj_size, markers));
    // watershed(dist, markers, mask = blb)
    BlobInfo b;
    TISEG_TRY(blobs_build(c, g, ImgMaskU8{blb}, par, rank, b, true));
    TISEG_TRY(ws_seed(c, g, markers, par, inst));
    TISEG_TRY(watershed_f64_dev(c, g, dist, par, rank, b, inst));
    return TISEG_OK;
}

// ---- scale_factor = 2 (the CoNIC config, hovernet_adam-lr1e-4_bs8_256x256_100e_conic.py:47) -----------------------
// cv2.resize(src, (0, 0), fx=2, fy=2) = bilinear with sample positions (d + 0.5) / 2 - 0.5: weights 0.75 / 0.25,
// clamped at the borders; horizontal pass, then vertical.  Arithmetic of the OpenCV 4.13 build the oracle runs
// (pinned in tests/cv_recipes.py): one-channel images with both sides >= 2 take OpenCV's 2x fast path, which
// interpolates as fma(a, x1 - x0, x0); everything else (two channels, degenerate sides) as x0 * (1 - a) + x1 * a.
__device__ __forceinline__ void up2_coord(int d, int n, int& s0, int& s1, float& a) {
    // f = (d + 0.5) * 0.5 - 0.5 = d / 2 - 0.25
    int s = (d & 1) ? (d >> 1) : (d >> 1) - 1;
    a = (d & 1) ? 0.25f : 0.75f;
    if (s < 0) { s = 0; a = 0.f; }
    if (s >= n - 1) { s = n - 1; a = 0.f; }
    s0 = s; s1 = min(s + 1, n - 1);
}
template <bool LERP>
__device__ __forceinline__ float up2_mix(float x0, float x1, float a) {
    if (LERP) return fmaf(a, __fsub_rn(x1, x0), x0);
    return __fadd_rn(__fmul_rn(x0, __fsub_rn(1.f, a)), __fmul_rn(x1, a));
}
template <class TI, int CN, bool LERP>
__global__ void __launch_bounds__(TISEG_THREADS)
k_resize_up2(Geom gd, int H, int W, const TI* __restrict__ src, float* __restrict__ dst) {
    Pix px;
    if (!warp_pixel(gd, px) || !px.ok) return;
    int y0, y1, x0, x1;
    float ay, ax;
    up2_coord(px.y, H, y0, y1, ay);
    up2_coord(px.x, W, x0, x1, ax);
    const TI* t = src + (long long)px.n * H * W * CN;
#pragma unroll
    for (int ch = 0; ch < CN; ++ch) {
        const float h0 = up2_mix<LERP>(to_f32(t[((long long)y0 * W + x0) * CN + ch]), to_f32(t[((long long)y0 * W + x1) * CN + ch]), ax);
        const float h1 = up2_mix<LERP>(to_f32(t[((long long)y1 * W + x0) * CN + ch]), to_f32(t[((long long)y1 * W + x1) * CN + ch]), ax);
        dst[(px.base + px.idx) * CN + ch] = up2_mix<LERP>(h0, h1, ay);
    }
}
// cv2.resize(labels, (W, H), interpolation=INTER_NEAREST) from (2H, 2W): source pixel (2y, 2x)
__global__ void __launch_bounds__(TISEG_THREADS)
k_resize_down2_nearest(Geom g, const int32_t* __restrict__ src, int32_t* __restrict__ dst) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    dst[px.base + px.idx] = src[(long long)px.n * g.P * 4 + (long long)(2 * px.y) * (2 * g.W) + 2 * px.x];
}

}  // namespace tiseg

using namespace tiseg;

template <class TI>
static int postproc_hover_entry(tiseg_ctx* c, const void* fore_map, const void* hv_map, const Geom& g, const Geom& gs,
                                int scale_factor, int ksize, int obj_size, int32_t* d_inst, uint8_t* d_blb, double* d_dist,
                                int32_t* d_mk) {
    const TI* d_fore = (const TI*)fore_map;
    const TI* d_hv = (const TI*)hv_map;
    if (scale_factor == 1) return postproc_hover_dev(c, g, d_fore, d_hv, ksize, obj_size, d_inst, d_blb, d_dist, d_mk);
    const size_t stotal = (size_t)gs.N * gs.P;
    float* fore2 = ws<float>(c, stotal);
    float* hv2 = ws<float>(c, stotal * 2);
    int32_t* inst2 = ws<int32_t>(c, stotal);
    if (!fore2 || !hv2 || !inst2) return TISEG_ERR_CUDA;
    const int H = g.H, W = g.W;
    if (H >= 2 && W >= 2) TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "(k_resize_up2<1, true>)"), (k_resize_up2<TI, 1, true>), warp_grid(gs), TISEG_THREADS, 0, gs, H, W, d_fore, fore2);
    else                  TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "(k_resize_up2<1, false>)"), (k_resize_up2<TI, 1, false>), warp_grid(gs), TISEG_THREADS, 0, gs, H, W, d_fore, fore2);
    TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "(k_resize_up2<2, false>)"), (k_resize_up2<TI, 2, false>), warp_grid(gs), TISEG_THREADS, 0, gs, H, W, d_hv, hv2);
    TISEG_TRY(postproc_hover_dev(c, gs, (const float*)fore2, (const float*)hv2, ksize, obj_size, inst2, d_blb, d_dist, d_mk));
    TISEG_LAUNCH(c, k_resize_down2_nearest, warp_grid(g), TISEG_THREADS, 0, g, inst2, d_inst);
    return TISEG_OK;
}

extern "C" int tiseg_postproc_hover_ex(tiseg_ctx* c, int dtype, const void* fore_map, const void* hv_map, int N, int H, int W,
                                       int scale_factor, int ksize, int obj_size, int32_t* inst_out, uint8_t* blb_out,
                                       double* dist_out, int32_t* marker_out) {
    TISEG_TRY(check_dtype(dtype, "tiseg_postproc_hover_ex"));
    if (!c || !fore_map || !hv_map || !inst_out) { set_error("tiseg_postproc_hover_ex: bad argument"); return TISEG_ERR_ARG; }
    if (scale_factor != 1 && scale_factor != 2) {
        set_error("tiseg_postproc_hover_ex: scale_factor must be 1 or 2 (the values of the reference configs), got " +
                  std::to_string(scale_factor));
        return TISEG_ERR_ARG;
    }
    if (ksize < 1 || ksize > 2 * SOBEL_RMAX + 1 || ksize % 2 == 0) {       // what cv2.Sobel refuses (and -1, Scharr)
        set_error("tiseg_postproc_hover_ex: ksize must be odd and in 1..31 (cv2.Sobel), got " + std::to_string(ksize));
        return TISEG_ERR_ARG;
    }
    if (obj_size < 0) {
        set_error("tiseg_postproc_hover_ex: obj_size must be >= 0, got " + std::to_string(obj_size));
        return TISEG_ERR_ARG;
    }
    TISEG_TRY(check_geom(N, H * scale_factor, W * scale_factor));
    begin_call(c);
    Geom g = make_geom(N, H, W);
    Geom gs = make_geom(N, H * scale_factor, W * scale_factor);          // the resolution the pipeline runs at
    size_t total = (size_t)N * g.P, stotal = (size_t)N * gs.P;
    const void* d_fore = in_ptr(c, fore_map, total * dtype_bytes(dtype));
    const void* d_hv = in_ptr(c, hv_map, total * 2 * dtype_bytes(dtype));
    int32_t* d_inst = tiseg::out(c, inst_out, total);
    uint8_t* d_blb = blb_out ? tiseg::out(c, blb_out, stotal) : nullptr;
    double* d_dist = dist_out ? tiseg::out(c, dist_out, stotal) : nullptr;
    int32_t* d_mk = marker_out ? tiseg::out(c, marker_out, stotal) : nullptr;
    if (!d_fore || !d_hv || !d_inst) return TISEG_ERR_CUDA;
    TISEG_TRY(with_dtype(dtype, [&](auto z) {
        return postproc_hover_entry<decltype(z)>(c, d_fore, d_hv, g, gs, scale_factor, ksize, obj_size, d_inst, d_blb, d_dist,
                                                 d_mk);
    }));
    return end_call(c);
}
