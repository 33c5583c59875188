// A8 — DIST postprocess: tiseg/models/segmentors/dist.py:275-284 -> dynamic_watershed_alias (:114-129)
// with prepare_prob (:31-40), H_reconstruction_erosion (:43-57; lambda = 0.0 => identity), find_maxima
// (:60-71), arrange_label (:101-111) and generate_wsl (:83-98).
//
//   d  = int32(clip(dist, 0, 255))             (truncation)             k_dist_prep (one pass: I, the mask plane,
//   I  = 255 - uint8(d);  b = d > 0.5  <=>  I < 255                      the marker candidates, the mask area)
//   markers = label(recon_by_erosion(min(255, I+1), I) - I, masked by b)
//           = 8-connected regional-minimum plateaus of I with value < 255, raster ids
//                                                                       bit-plane CCL of the candidates + rank
//   ws = watershed(I, markers, mask=b)                                   K6 (bucket flood)
//   arranged = label(ws, background = most frequent value of ws)         k_ws_hist + k_pick_bg + CCL
//   arranged[3x3 window holds >= 2 different non-zero labels] = 0        k_wsl_remove
#include "ccl.cuh"
#include "watershed.cuh"

namespace tiseg {

// ---- the front: level image, mask plane, marker candidates --------------------------------------------------------------
// Regional-minimum plateaus without labelling every plateau of the image.  A pixel is a CANDIDATE if its value is
// below 255 and no 8-neighbour is strictly lower.  A plateau P (maximal 8-connected set of equal values) is a regional
// minimum iff all its pixels are candidates.  Label the candidates only (equal value, 8-connected): if P is a
// minimum it comes out as one component, none of whose pixels has an equal-valued non-candidate neighbour; if P is
// not, every candidate component C inside it is a proper subset of the connected P, so some pixel of C touches an
// equal-valued pixel outside C — which must be a non-candidate (a candidate would have joined C).  Hence:
// minimum plateaus = candidate components without an "equal-valued non-candidate neighbour" flag.  On a distance map
// the candidates are the few pixels around each nucleus centre.
// Candidates are a few percent of the pixels, so the plateau labelling works on one 32-bit word per 32-pixel row
// segment (bits[n, y, seg]).  Adjacent candidates always carry the same level (the higher one would have a lower
// neighbour), so the labelling is binary.
//   k_dist_prep            one pass over the distance map: level image I, mask plane, candidate bitmap, bitmap of the
//                          candidates that touch an equal-valued non-candidate, mask pixels per tile
//   (lambda > 0)           k_dist_prep without the candidates; k_plateau_bits takes them from the reconstructed image
//   bitccl_build           8-connected components of the candidate bitmap (bitccl.cuh: union-find over runs)
//   (bitccl_build)         low[root] = 1 for plateaus with a bad pixel; k_filter_root_bits drops them from the roots
//   k_marker_scatter       the seed map (rank of the plateau's root on its pixels; zero elsewhere by memset)
__device__ __forceinline__ int run_len_from(unsigned w, int a) {       // length of the run of ones starting at bit a
    const unsigned x = w >> a;
    return x == 0xffffffffu ? 32 : __ffs(~x) - 1;
}
__device__ __forceinline__ int run_start_of(unsigned w, int q) {       // first bit of the run of ones containing bit q
    const unsigned below = ~w & ((1u << q) - 1u);
    return below ? 32 - __clz(below) : 0;
}

// dist.py:277-279 and 116: d = int32(clip(dist, 0, 255)) (truncation), I = 255 - uint8(d).  The comparison is false
// for NaN, like numpy's, so NaN passes the upper clip; the unsigned truncating conversion then gives 0 for NaN and for
// every negative value (the lower clip), so NaN is level 255 (outside the mask b = d > 0.5 = I < 255).  Three
// instructions per pixel in this issue-bound pass, against five for an explicit lower clip and a signed conversion.
__device__ __forceinline__ unsigned dist_level(float v) {
    if (v > 255.f) v = 255.f;
    return 255u - __float2uint_rz(v);
}

// The walk.  One warp = a 128-column strip x FR_BAND rows walking down, four pixels per thread and row.  Both bitmaps are
// 3x3 minima: with J = I where a pixel is NOT a candidate and 255 where it is, a candidate p touches an equal-valued
// non-candidate iff min3x3(J)(p) == I(p) (every neighbour of a candidate is >= it).  A thread holds its four pixels as
// two u16x2 words (pixels 0,1 / 2,3) so that a three-way minimum of two pixels is ONE instruction (VIMNMX3.U16x2,
// __vimin3_u16x2); the warp keeps the last row minima in registers and takes left / right pixels from the neighbouring
// lanes.  The stencil of a stencil needs two pixels beyond the strip on each side: lanes 0 and 31 load them (one pair per
// row), compute the candidate flag of the column next to the strip with a scalar copy of the stencil, and hand its level
// (I) and its J to their own horizontal minima.  The band is walked from two rows above it to two rows below it, so the
// vertical halo costs 4 / FR_BAND of the loads.  Pixels outside the image are level 255: never lower than a neighbour,
// never a candidate, never in the mask, so every bit beyond W stays zero.
#define FR_BAND 64
#define FR_AHEAD 2               // rows of loads in flight per thread
struct Px4 { unsigned lo, hi; };                      // (px0 | px1 << 16), (px2 | px3 << 16)
// horizontal 3-minimum; `edge` = the value of the column beyond the strip (used by lanes 0 and 31)
__device__ __forceinline__ Px4 fr_hmin(Px4 v, int lane, unsigned edge) {
    unsigned hl = __shfl_up_sync(0xffffffffu, v.hi, 1);                        // pixels 2,3 of the thread to the left
    unsigned lr = __shfl_down_sync(0xffffffffu, v.lo, 1);                      // pixels 0,1 of the thread to the right
    if (lane == 0) hl = edge << 16;
    if (lane == 31) lr = edge;
    const unsigned a = __byte_perm(hl, v.lo, 0x5432);                          // (px-1, px0)
    const unsigned m = __byte_perm(v.lo, v.hi, 0x5432);                        // (px1, px2)
    const unsigned z = __byte_perm(v.hi, lr, 0x5432);                          // (px3, px4)
    Px4 r;
    r.lo = __vimin3_u16x2(a, v.lo, m);
    r.hi = __vimin3_u16x2(m, v.hi, z);
    return r;
}
// per 16-bit lane (values <= 255): 1 where the lane is non-zero
__device__ __forceinline__ unsigned pb_nonzero(unsigned x) { return ((x + 0x7fff7fffu) >> 15) & 0x00010001u; }
// flags at bits 0 / 16 of (lo, hi) -> 4-bit nibble, bit k = pixel k
__device__ __forceinline__ unsigned pb_nibble(unsigned lo, unsigned hi) {
    const unsigned t = lo | (hi << 2);
    return (t | (t >> 15)) & 15u;
}

// The sources of the walk.  issue() starts the loads of row y (nothing outside the image); levels() turns them into the
// thread's four levels (byte k = pixel k) and the pair beyond the strip edge (byte 0 = column xe, byte 1 = xe + 1).
// VEC: W % 4 == 0 and the rows are aligned to four elements, so a thread's four pixels are in the row or out of it as a
// whole, and the edge pair (at an even column) is aligned to two.
// The distance map, fp32 / fp16 / bf16, converted to fp32 at the load.
template <class TI, bool VEC>
struct DistSrc {
    static constexpr bool vec = VEC;
    struct Raw { float d[4], e[2]; };
    const TI* t;
    __device__ __forceinline__ void issue(const Geom& g, int y, int x, int xe, bool oke, Raw& r) const {
        r.d[0] = r.d[1] = r.d[2] = r.d[3] = 0.f;                      // (0 is level 255)
        r.e[0] = r.e[1] = 0.f;
        if (y < 0 || y >= g.H) return;                                // (uniform)
        const int ro = y * g.W;
        if (VEC) {
            if (x < g.W) ld4f_aligned(t + ro + x, r.d);
            if (oke) {
                const float2 f = to_f32(*reinterpret_cast<const typename Pair<TI>::type*>(t + ro + xe));
                r.e[0] = f.x; r.e[1] = f.y;
            }
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k) if (x + k < g.W) r.d[k] = to_f32(t[ro + x + k]);
            if (oke) r.e[0] = to_f32(t[ro + xe]);
            if (oke && xe + 1 < g.W) r.e[1] = to_f32(t[ro + xe + 1]);
        }
    }
    __device__ __forceinline__ void levels(const Raw& r, unsigned& p, unsigned& e) const {
        p = dist_level(r.d[0]) | (dist_level(r.d[1]) << 8) | (dist_level(r.d[2]) << 16) | (dist_level(r.d[3]) << 24);
        e = dist_level(r.e[0]) | (dist_level(r.e[1]) << 8);
    }
};
// A level image (u8), read as it is.
template <bool VEC>
struct LevelSrc {
    static constexpr bool vec = VEC;
    struct Raw { unsigned p, e; };
    const uint8_t* t;
    __device__ __forceinline__ void issue(const Geom& g, int y, int x, int xe, bool oke, Raw& r) const {
        r.p = 0xffffffffu; r.e = 0xffffu;
        if (y < 0 || y >= g.H) return;                                // (uniform)
        const uint8_t* row = t + y * g.W;
        if (VEC) {
            if (x < g.W) r.p = *reinterpret_cast<const unsigned*>(row + x);
        } else {
            unsigned p = 0u;
#pragma unroll
            for (int k = 0; k < 4; ++k) p |= (x + k < g.W ? (unsigned)row[x + k] : 255u) << (8 * k);
            r.p = p;
        }
        if (oke) r.e = row[xe] | ((xe + 1 < g.W ? (unsigned)row[xe + 1] : 255u) << 8);
    }
    __device__ __forceinline__ void levels(const Raw& r, unsigned& p, unsigned& e) const { p = r.p; e = r.e; }
};

// LEVELS: store I (It) and the mask plane (mt) of rows [y0, y1) and add the band's mask pixels to *marea.
// STENCIL: the candidate (cb) and bad-candidate (bb) bitmaps of rows [y0, y1).
template <bool LEVELS, bool STENCIL, class Src>
__device__ __forceinline__ void fr_walk(const Geom& g, const Src& src, uint8_t* __restrict__ It, unsigned* __restrict__ mt,
                                        unsigned* __restrict__ cb, unsigned* __restrict__ bb, int* __restrict__ marea,
                                        int lane, int x0, int y0, int y1) {
    const int W = g.W, x = x0 + lane * 4;
    const int xe = lane == 0 ? x0 - 2 : x0 + 128;                       // the pair beyond the strip edge
    const bool oke = STENCIL && ((lane == 0 && x0 > 0) || (lane == 31 && xe < W));
    const int seg = (x0 >> 5) + (lane >> 3);
    const bool cwriter = (lane & 7) == 0 && seg < g.SEG, mwriter = (lane & 7) == 4 && seg < g.SEG;
    const int q = (lane & 3) * 4;
    const int ylo = STENCIL ? y0 - 2 : y0, yhi = STENCIL ? y1 + 2 : y1;
    const Px4 FF = {0x00ff00ffu, 0x00ff00ffu};
    Px4 hI1 = FF, hI2 = FF;          // row minima of I, rows r-1 and r-2
    Px4 hJ1 = FF, hJ2 = FF;          // row minima of J, rows r-2 and r-3
    Px4 I1 = FF, I2 = FF;            // I of rows r-1, r-2
    Px4 C2 = {0u, 0u};               // candidate flags (bits 0 / 16) of row r-2
    unsigned eh1 = 255u, eh2 = 255u, en1 = 255u;   // lanes 0 / 31, the column beyond the edge: row minima (r-1, r-2), I (r-1)
    int area = 0;
    typename Src::Raw raw[FR_AHEAD];
    int yn = ylo;
    auto issue = [&](typename Src::Raw& r) { src.issue(g, yn < yhi ? yn : -1, x, xe, oke, r); ++yn; };
#pragma unroll
    for (int u = 0; u < FR_AHEAD; ++u) issue(raw[u]);
    for (int r0 = ylo; r0 < yhi; r0 += FR_AHEAD) {
        unsigned pv[FR_AHEAD], ev[FR_AHEAD];
#pragma unroll
        for (int u = 0; u < FR_AHEAD; ++u) src.levels(raw[u], pv[u], ev[u]);
        if (r0 + FR_AHEAD < yhi) {                                      // (uniform) always FR_AHEAD rows ahead
#pragma unroll
            for (int u = 0; u < FR_AHEAD; ++u) issue(raw[u]);
        }
#pragma unroll
        for (int u = 0; u < FR_AHEAD; ++u) {
            const int r = r0 + u;                                       // (rows past yhi: 255, nothing emitted)
            const unsigned p = pv[u];
            Px4 c;
            c.lo = __byte_perm(p, 0u, 0x4140);
            c.hi = __byte_perm(p, 0u, 0x4342);
            const bool lrow = LEVELS && r >= y0 && r < y1;              // (uniform)
            unsigned mn = 0u;
            if (LEVELS) {
                if (lrow) {
                    uint8_t* dst = It + r * W + x;
                    if (Src::vec) { if (x < W) *reinterpret_cast<unsigned*>(dst) = p; }
                    else {
#pragma unroll
                        for (int k = 0; k < 4; ++k) if (x + k < W) dst[k] = (uint8_t)(p >> (8 * k));
                    }
                }
                mn = pb_nibble(pb_nonzero(c.lo ^ 0x00ff00ffu), pb_nonzero(c.hi ^ 0x00ff00ffu));
            }
            unsigned cn = 0u, bn = 0u;
            if (STENCIL) {
                const unsigned e = ev[u];
                const unsigned en = lane == 0 ? e >> 8 : e & 255u;     // the column next to the strip
                const unsigned eh0 = min(min(e & 255u, e >> 8), lane == 0 ? c.lo & 0xffffu : c.hi >> 16);
                const Px4 hI0 = fr_hmin(c, lane, en);
                // candidates of row r-1: the 3x3 minimum (centre included) equals the pixel, and the pixel is below 255
                Px4 C1, J;
                {
                    const unsigned mlo = __vimin3_u16x2(hI0.lo, hI1.lo, hI2.lo), mhi = __vimin3_u16x2(hI0.hi, hI1.hi, hI2.hi);
                    const unsigned nlo = pb_nonzero(I1.lo - mlo) | (((I1.lo + 0x00010001u) >> 8) & 0x00010001u);
                    const unsigned nhi = pb_nonzero(I1.hi - mhi) | (((I1.hi + 0x00010001u) >> 8) & 0x00010001u);
                    C1.lo = nlo ^ 0x00010001u;
                    C1.hi = nhi ^ 0x00010001u;
                    J.lo = I1.lo | (C1.lo * 255u);
                    J.hi = I1.hi | (C1.hi * 255u);
                }
                const unsigned eJ = (min(min(eh0, eh1), eh2) == en1 && en1 < 255u) ? 255u : en1;
                const Px4 hJ0 = fr_hmin(J, lane, eJ);
                // bad candidates of row r-2
                const unsigned jlo = __vimin3_u16x2(hJ0.lo, hJ1.lo, hJ2.lo), jhi = __vimin3_u16x2(hJ0.hi, hJ1.hi, hJ2.hi);
                const unsigned Blo = C2.lo & ~pb_nonzero(jlo ^ I2.lo), Bhi = C2.hi & ~pb_nonzero(jhi ^ I2.hi);
                cn = pb_nibble(C2.lo, C2.hi);
                bn = pb_nibble(Blo, Bhi);
                hI2 = hI1; hI1 = hI0; hJ2 = hJ1; hJ1 = hJ0; I2 = I1; I1 = c; C2 = C1;
                eh2 = eh1; eh1 = eh0; en1 = en;
            }
            // eight lanes x four pixels -> one 32-bit word of each map: lanes 0..3 of a group fill the low half-words, lanes
            // 4..7 the high ones; lane 0 of the group stores the candidate words (row r-2), lane 4 the mask word (row r)
            unsigned w = (cn | (bn << 16)) << q, m = mn << q;
            if (STENCIL) { w |= __shfl_xor_sync(0xffffffffu, w, 1); w |= __shfl_xor_sync(0xffffffffu, w, 2); }
            if (LEVELS) { m |= __shfl_xor_sync(0xffffffffu, m, 1); m |= __shfl_xor_sync(0xffffffffu, m, 2); }
            const unsigned o = __shfl_xor_sync(0xffffffffu, (lane & 4) ? w : m, 4);
            const int y = r - 2;
            if (STENCIL && y >= y0 && y < y1 && cwriter) {
                cb[y * g.SEG + seg] = (w & 0xffffu) | (o << 16);
                bb[y * g.SEG + seg] = (w >> 16) | (o & 0xffff0000u);
            }
            if (lrow && mwriter) {
                const unsigned mw = o | (m << 16);
                mt[r * g.SEG + seg] = mw;
                area += __popc(mw);
            }
        }
    }
    if (LEVELS) {
        area = __reduce_add_sync(0xffffffffu, area);
        if (lane == 0 && area) atomicAdd(marea, area);
    }
}

// warp -> (strip, band) of tile blockIdx.y; false for the warps past the last band
__device__ __forceinline__ bool fr_warp(const Geom& g, int& x0, int& y0, int& y1) {
    const int strips = (g.W + 127) >> 7, bands = (g.H + FR_BAND - 1) / FR_BAND;
    const long long wi = (long long)blockIdx.x * TISEG_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    if (wi >= (long long)strips * bands) return false;
    const int band = (int)(wi / strips), strip = (int)(wi - (long long)band * strips);
    x0 = strip * 128; y0 = band * FR_BAND; y1 = min(y0 + FR_BAND, g.H);
    return true;
}
inline dim3 fr_grid(const Geom& g) {
    const long long warps = (long long)((g.W + 127) >> 7) * ((g.H + FR_BAND - 1) / FR_BAND);
    return dim3((unsigned)((warps + TISEG_WARPS_PER_BLOCK - 1) / TISEG_WARPS_PER_BLOCK), (unsigned)g.N);
}

// the distance map -> I, the mask plane, marea (zeroed beforehand) and, with STENCIL, the candidate / bad-candidate planes.
// (three blocks per SM at 80 registers, two rows ahead: 0.140 ms per 64 x 1000^2 step on a B200 at 1000 W.  Measured slower
//  there: four rows ahead at 106 registers, two blocks per SM (+24 %); four blocks per SM with spills (+30 %); bands of 32,
//  128 or 168 rows instead of 64 (+5 to +12 %).  The pass is bound by instruction issue.)
template <class TI, bool STENCIL>
__global__ void __launch_bounds__(TISEG_THREADS, 3)
k_dist_prep(Geom g, const TI* __restrict__ dist, uint8_t* __restrict__ I, unsigned* __restrict__ mbits, unsigned* __restrict__ cbits,
            unsigned* __restrict__ bbits, int* __restrict__ marea, bool vec) {
    int x0, y0, y1;
    if (!fr_warp(g, x0, y0, y1)) return;
    const int lane = threadIdx.x & 31, n = blockIdx.y;
    // (tile bases as opaque register pairs + 32-bit offsets: one IMAD.WIDE per access in this issue-bound loop)
    const TI* dt = dist + (long long)n * g.P;
    uint8_t* It = I + (long long)n * g.P;
    unsigned* mt = mbits + (long long)n * g.H * g.SEG;
    unsigned* ct = STENCIL ? cbits + (long long)n * g.H * g.SEG : nullptr;
    unsigned* bt = STENCIL ? bbits + (long long)n * g.H * g.SEG : nullptr;
    asm volatile("" : "+l"(dt)); asm volatile("" : "+l"(It)); asm volatile("" : "+l"(mt));
    __builtin_assume(__isGlobal(dt)); __builtin_assume(__isGlobal(It)); __builtin_assume(__isGlobal(mt));
    if (STENCIL) {
        asm volatile("" : "+l"(ct)); asm volatile("" : "+l"(bt));
        __builtin_assume(__isGlobal(ct)); __builtin_assume(__isGlobal(bt));
    }
    if (vec) fr_walk<true, STENCIL>(g, DistSrc<TI, true>{dt}, It, mt, ct, bt, marea + n, lane, x0, y0, y1);
    else fr_walk<true, STENCIL>(g, DistSrc<TI, false>{dt}, It, mt, ct, bt, marea + n, lane, x0, y0, y1);
}

// the candidate / bad-candidate planes of a level image (the H-reconstruction of I when lambda > 0)
__global__ void __launch_bounds__(TISEG_THREADS)
k_plateau_bits(Geom g, const uint8_t* __restrict__ I, unsigned* __restrict__ cbits, unsigned* __restrict__ bbits, bool vec) {
    int x0, y0, y1;
    if (!fr_warp(g, x0, y0, y1)) return;
    const int lane = threadIdx.x & 31, n = blockIdx.y;
    const uint8_t* It = I + (long long)n * g.P;
    unsigned* ct = cbits + (long long)n * g.H * g.SEG;
    unsigned* bt = bbits + (long long)n * g.H * g.SEG;
    asm volatile("" : "+l"(It)); asm volatile("" : "+l"(ct)); asm volatile("" : "+l"(bt));
    __builtin_assume(__isGlobal(It)); __builtin_assume(__isGlobal(ct)); __builtin_assume(__isGlobal(bt));
    if (vec) fr_walk<false, true>(g, LevelSrc<true>{It}, nullptr, nullptr, ct, bt, nullptr, lane, x0, y0, y1);
    else fr_walk<false, true>(g, LevelSrc<false>{It}, nullptr, nullptr, ct, bt, nullptr, lane, x0, y0, y1);
}

// seeds: rank of the plateau's root on the pixels of every run of a minimum plateau (the map is zeroed beforehand).  Every
// seed run also reports to the blob of the mask it lies in: the blob's marker label range (lmin / lmax: one label = the blob
// is simply filled) and, at the seed pixels, the blob id the flood's staging compares with (a run is 4-connected: one blob)
__global__ void __launch_bounds__(TISEG_THREADS)
k_marker_scatter(Geom g, const unsigned* __restrict__ bits, const int* __restrict__ par, const uint8_t* __restrict__ low,
                 const int* __restrict__ rank, int32_t* __restrict__ markers, BitPlanes mask, const int* __restrict__ bpar,
                 const int* __restrict__ brank, BlobInfo b, int* __restrict__ seed_blob, unsigned* __restrict__ seed_bits) {
    const long long words = (long long)g.H * g.SEG;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= words) return;
    const int n = blockIdx.y;
    unsigned w = bits[(long long)n * words + t];
    if (!w) { seed_bits[(long long)n * words + t] = 0u; return; }
    unsigned smask = 0u;
    const int y = (int)(t / g.SEG), seg = (int)(t - (long long)y * g.SEG);
    const long long base = (long long)n * g.P;
    const int idx0 = y * g.W + seg * 32;
    while (w) {
        const int a = __ffs(w) - 1, len = run_len_from(w, a);
        w = len == 32 ? 0u : w & ~(((1u << len) - 1u) << a);
        const int root = find_ro(par + base, bit_node_of(BitPlanes{bits, nullptr, nullptr, nullptr, nullptr}, g, (long long)n * words, y,
                                                           seg * 32 + a));
        if (low[base + root]) continue;
        const int id = rank[base + root];
        const int bid = blob_id_at(mask, g, n, bpar, brank, y, seg * 32 + a);
        const long long o = (long long)n * b.KS + bid;
        atomicMin(&b.lmin[o], id);
        atomicMax(&b.lmax[o], id);
        for (int k = 0; k < len; ++k) { markers[base + idx0 + a + k] = id; seed_blob[base + idx0 + a + k] = bid; }
        smask |= len == 32 ? 0xffffffffu : (((1u << len) - 1u) << a);
    }
    seed_bits[(long long)n * words + t] = smask;
}

// clear, in the bitmap of the roots that ccl_flatten left, the roots whose component is not a minimum plateau
__global__ void __launch_bounds__(TISEG_THREADS)
k_filter_root_bits(Geom g, const uint8_t* __restrict__ low, unsigned* bits) {
    const long long words = (long long)g.H * g.SEG;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= words) return;
    const int n = blockIdx.y;
    unsigned m = bits[(long long)n * words + t];
    if (!m) return;
    const int y = (int)(t / g.SEG), seg = (int)(t - (long long)y * g.SEG);
    unsigned keep = m;
    while (m) {
        const int b = __ffs(m) - 1;
        m &= m - 1;
        if (low[(long long)n * g.P + (long long)y * g.W + seg * 32 + b]) keep &= ~(1u << b);
    }
    bits[(long long)n * words + t] = keep;
}

// histogram of the flood labels (values 0..K) and the first raster pixel of each label, one pair of atomics per
// in-segment run
template <bool LISTED>
__global__ void __launch_bounds__(TISEG_THREADS)
k_ws_hist(Geom g, const int32_t* __restrict__ ws, int* hist, int* first, int KS, bool vec) {
    Quad q;
    if (!warp_quad(g, q)) return;
    FOR_TILES(LISTED, g, n) {
        q.n = n; q.base = (long long)n * g.P;
        int v[4];
        quad_load_i32(g, q, ws + q.base, 0, vec, v);
        // label 0 (the background, by far the longest runs) is not counted: its total is P minus the others
        if (!__any_sync(0xffffffffu, (v[0] | v[1] | v[2] | v[3]) != 0)) continue;
        const QuadRuns r = quad_runs(v, 0, q.lane);
        FOR_QUAD_RUNS(r, k, len) {
            const long long o = (long long)q.n * KS + v[k];
            atomicAdd(&hist[o], (int)len);
            atomicMin(&first[o], q.y * g.W + q.x + (int)k);
        }
    }
}

__global__ void k_init_label_tables(int* hist, int* first, int KS, const int* __restrict__ counts) {
    int n = blockIdx.y;
    int k = counts[n];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i <= k; i += gridDim.x * blockDim.x) {
        hist[(long long)n * KS + i] = 0;
        first[(long long)n * KS + i] = INT_MAX;
    }
}

// arrange_label's background: np.unique(return_counts) + argmax => the most frequent value, smallest value on ties.
// Tiles whose background is NOT 0 (one flood region larger than everything unlabelled) go on the list of the
// general relabelling path.
// A flood label covers at most the mask and the value 0 at least its complement, so with a mask of at most half the tile
// the background of arrange_label is 0 without counting anything (ties go to the smallest value).  Only denser tiles go on
// the list of the histogram pass.
__global__ void k_dense_tiles(const int* __restrict__ marea, int N, int P, int* bg, int* dense, int* ndense) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    bg[n] = 0;
    if (2ll * marea[n] > (long long)P) dense[atomicAdd(ndense, 1)] = n;
}

__global__ void k_pick_bg(const int* __restrict__ hist, int KS, const int* __restrict__ counts, int P, int* bg,
                          int* flagged, int* nflagged, const int* __restrict__ dense, const int* __restrict__ ndense) {
    __shared__ unsigned long long s[256];
    __shared__ long long tot[256];
    if (dense && (int)blockIdx.x >= *ndense) return;
    int n = dense ? dense[blockIdx.x] : blockIdx.x;
    int k = counts[n];
    // key = (count << 32) | (0xffffffff - value): max key = largest count, then smallest value
    unsigned long long best = 0;
    long long sum = 0;
    for (int v = 1 + threadIdx.x; v <= k; v += blockDim.x) {
        unsigned cnt = (unsigned)hist[(long long)n * KS + v];
        sum += cnt;
        unsigned long long key = ((unsigned long long)cnt << 32) | (0xffffffffu - (unsigned)v);
        if (key > best) best = key;
    }
    s[threadIdx.x] = best;
    tot[threadIdx.x] = sum;
    __syncthreads();
    for (int d = 128; d; d >>= 1) {
        if (threadIdx.x < d) {
            if (s[threadIdx.x + d] > s[threadIdx.x]) s[threadIdx.x] = s[threadIdx.x + d];
            tot[threadIdx.x] += tot[threadIdx.x + d];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        unsigned long long zero_key = ((unsigned long long)(unsigned)(P - tot[0]) << 32) | 0xffffffffu;   // value 0
        unsigned long long w = zero_key > s[0] ? zero_key : s[0];
        int b = (int)(0xffffffffu - (unsigned)(w & 0xffffffffu));
        bg[n] = b;
        if (b != 0) flagged[atomicAdd(nflagged, 1)] = n;
    }
}

// Fast relabelling when the background is 0.  Every flood region is one 8-connected component (its marker plateau is
// 8-connected and the flood grows it by 4-neighbours), so label(ws) only renumbers the regions by their first
// raster pixel: set the bit of each region's first pixel, rank the bitmap, look the ids up.
__global__ void k_first_bits(Geom g, const int* __restrict__ first, int KS, const int* __restrict__ counts, unsigned* bits) {
    int n = blockIdx.y;
    int k = counts[n];
    for (int l = 1 + blockIdx.x * blockDim.x + threadIdx.x; l <= k; l += gridDim.x * blockDim.x) {
        int idx = first[(long long)n * KS + l];
        if (idx == INT_MAX) continue;
        int y = idx / g.W, x = idx - y * g.W;
        atomicOr(&bits[((long long)n * g.H + y) * g.SEG + (x >> 5)], 1u << (x & 31));
    }
}
__global__ void k_arrange_lut(Geom g, const int* __restrict__ first, const int* __restrict__ rank, int KS,
                              const int* __restrict__ counts, int* __restrict__ lut) {
    int n = blockIdx.y;
    int k = counts[n];
    for (int l = blockIdx.x * blockDim.x + threadIdx.x; l <= k; l += gridDim.x * blockDim.x) {
        int idx = l ? first[(long long)n * KS + l] : INT_MAX;
        lut[(long long)n * KS + l] = idx == INT_MAX ? 0 : rank[(long long)n * g.P + idx];
    }
}

// generate_wsl + "arranged[wsl > 0] = 0" (dist.py:83-98, 128): a pixel whose 3x3 window holds another non-zero label is a
// watershed line.  `lut` (may be null): the id of each label value, applied to the pixels that survive.
// `mask` (may be null): F plane of the pixels of `lab` that carry a value — everything else counts as 0 whatever the map
// holds there (the flood output is only ever written inside the mask b, so the label map needs no zero fill).
// One warp = a 128-column strip x WR_BAND rows walking down, four pixels per thread (one 128-bit load per row).  With u = label - 1 as unsigned (0 -> 0xffffffff) "another non-zero
// label in the window" is  max3x3(label) != v  or  umin3x3(u) != v - 1,  and both are separable: the row aggregates of
// the last two rows stay in registers, the horizontal neighbours come from the adjacent lanes (the strip's outer columns
// from one extra load in lanes 0 / 31).  Every row is loaded once; the earlier version (a 3x3 window per thread: three row
// loads + six scalar loads) ran at half the HBM rate (profiles/r2_*).
#define WR_BAND 32
#define WR_AHEAD 4               // rows of loads in flight per thread
struct WrAgg { int hx[4]; unsigned hn[4]; };                 // per pixel: max / (unsigned) min of (label - 1) over the row's 3 columns
__device__ __forceinline__ void wr_agg(const int (&v)[4], int e, int lane, WrAgg& a) {
#pragma unroll
    for (int k = 0; k < 4; ++k) { a.hx[k] = 0; a.hn[k] = ~0u; }
    if (__any_sync(0xffffffffu, (v[0] | v[1] | v[2] | v[3] | e) != 0)) {       // (uniform)
        int c[6];
        c[0] = __shfl_up_sync(0xffffffffu, v[3], 1);
        c[5] = __shfl_down_sync(0xffffffffu, v[0], 1);
        if (lane == 0) c[0] = e;
        if (lane == 31) c[5] = e;
        c[1] = v[0]; c[2] = v[1]; c[3] = v[2]; c[4] = v[3];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            a.hx[k] = max(max(c[k], c[k + 1]), c[k + 2]);
            a.hn[k] = min(min((unsigned)(c[k] - 1), (unsigned)(c[k + 1] - 1)), (unsigned)(c[k + 2] - 1));
        }
    }
}
// the finished row: v with the aggregates of the rows above (a2), of its own row (a1) and below (a0)
template <bool FULL, bool LUT>
__device__ __forceinline__ void wr_emit(const int (&v)[4], const WrAgg& a2, const WrAgg& a1, const WrAgg& a0, const int* __restrict__ tl,
                                        int32_t* __restrict__ dst, int x, int W) {
    int o[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int M = max(max(a2.hx[k], a1.hx[k]), a0.hx[k]);
        const unsigned m = min(min(a2.hn[k], a1.hn[k]), a0.hn[k]);
        const bool keep = M == v[k] && m == (unsigned)(v[k] - 1);          // (false for v = 0: m <= 0xffffffff - ... never v - 1 = ~0u with M == 0 unless all zero)
        o[k] = keep ? v[k] : 0;
    }
    if (LUT) {
        if (o[0] | o[1] | o[2] | o[3]) {
#pragma unroll
            for (int k = 0; k < 4; ++k) o[k] = tl[o[k]];                   // (lut[0] = 0)
        }
    }
    if (FULL) *reinterpret_cast<int4*>(dst) = make_int4(o[0], o[1], o[2], o[3]);
    else {
#pragma unroll
        for (int k = 0; k < 4; ++k) if (x + k < W) dst[k] = o[k];
    }
}
// a row as it comes from memory: the thread's four labels, its mask word, and (lanes 0 / 31) the strip's outer neighbour with
// the mask word that covers it.  The labels are loaded whether or not the mask has them (the values are discarded in
// wr_finish): a load that waits for the mask word doubles the latency chain of this latency-bound walk.
struct WrRaw { int q[4]; unsigned mw, mew; int e; };
template <bool FULL, bool MASKED>
__device__ __forceinline__ void wr_issue(const int32_t* __restrict__ tile, const unsigned* __restrict__ mt, int y, int H, int po, int eo,
                                         int mo, int meo, bool hasw, bool oke, int x, int W, WrRaw& r) {
    r.q[0] = r.q[1] = r.q[2] = r.q[3] = 0; r.mw = 0u; r.mew = 0u; r.e = 0;
    if (y >= 0 && y < H) {                       // (uniform)
        if (MASKED) {
            if (hasw) r.mw = mt[mo];
            if (oke) r.mew = mt[meo];
        }
        if (FULL) { const int4 t = *reinterpret_cast<const int4*>(tile + po); r.q[0] = t.x; r.q[1] = t.y; r.q[2] = t.z; r.q[3] = t.w; }
        else {
#pragma unroll
            for (int k = 0; k < 4; ++k) if (x + k < W) r.q[k] = tile[po + k];
        }
        if (oke) r.e = tile[eo];
    }
}
template <bool MASKED>
__device__ __forceinline__ void wr_finish(const WrRaw& r, int sh, int eb, int (&v)[4], int& e) {
    if (MASKED) {
        const unsigned nib = r.mw >> sh;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            v[k] = r.q[k];
            asm("{\n\t.reg .pred p;\n\t.reg .b32 t;\n\tand.b32 t, %1, %2;\n\tsetp.ne.u32 p, t, 0;\n\tselp.s32 %0, %0, 0, p;\n\t}"
                : "+r"(v[k]) : "r"(nib), "r"(1u << k));
        }
        e = (r.mew >> eb) & 1u ? r.e : 0;
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) v[k] = r.q[k];
        e = r.e;
    }
}
template <bool FULL, bool MASKED, bool LUT>
__device__ __forceinline__ void wr_strip(const Geom& g, const int32_t* __restrict__ tile, const unsigned* __restrict__ mt,
                                         const int* __restrict__ tl, int32_t* __restrict__ otile, int lane, int x, int y0, int y1) {
    const int W = g.W, SEG = g.SEG, H = g.H;
    const int xe = lane == 0 ? x - 1 : x + 4;
    const bool oke = (lane == 0 || lane == 31) && xe >= 0 && xe < W;
    const bool hasw = (x >> 5) < SEG;
    const int sh = (lane & 7) * 4, eb = xe & 31;
    // the next row to load and the 32-bit offsets of this thread's pixels / mask words in it (tile-local: P < 2^30)
    int yn = y0 - 1, po = yn * W + x, eo = yn * W + xe, mo = yn * SEG + (x >> 5), meo = yn * SEG + (xe >> 5);
    auto issue = [&](WrRaw& r) {
        wr_issue<FULL, MASKED>(tile, mt, yn, H, po, eo, mo, meo, hasw, oke, x, W, r);
        ++yn; po += W; eo += W; mo += SEG; meo += SEG;
    };
    int oo = y0 * W + x;                         // offset of the next output row
    WrAgg a2, a1, a0;
    int v1[4], v0[4], e;
    WrRaw r[WR_AHEAD];
    issue(r[0]); issue(r[1]);                    // rows y0 - 1 (zeros outside the image) and y0
    wr_finish<MASKED>(r[0], sh, eb, v0, e);
    wr_agg(v0, e, lane, a2);
    wr_finish<MASKED>(r[1], sh, eb, v1, e);
    wr_agg(v1, e, lane, a1);
#pragma unroll
    for (int u = 0; u < WR_AHEAD; ++u) issue(r[u]);       // always WR_AHEAD rows ahead of the arithmetic
    int y = y0;
    for (; y + WR_AHEAD <= y1; y += WR_AHEAD) {  // rows y + 1 .. y + WR_AHEAD complete rows y .. y + WR_AHEAD - 1
        int v[WR_AHEAD][4], ee[WR_AHEAD];
#pragma unroll
        for (int u = 0; u < WR_AHEAD; ++u) wr_finish<MASKED>(r[u], sh, eb, v[u], ee[u]);
        if (y + WR_AHEAD < y1) {                 // (rows beyond y1 are never used)
#pragma unroll
            for (int u = 0; u < WR_AHEAD; ++u) issue(r[u]);
        }
#pragma unroll
        for (int u = 0; u < WR_AHEAD; ++u) {
            wr_agg(v[u], ee[u], lane, a0);
            wr_emit<FULL, LUT>(v1, a2, a1, a0, tl, otile + oo, x, W);
            oo += W;
            a2 = a1; a1 = a0;
#pragma unroll
            for (int k = 0; k < 4; ++k) v1[k] = v[u][k];
        }
    }
#pragma unroll
    for (int u = 0; u < WR_AHEAD - 1; ++u) {     // (the rest of a short band: r[u] holds row y + 1)
        if (y < y1) {
            wr_finish<MASKED>(r[u], sh, eb, v0, e);
            wr_agg(v0, e, lane, a0);
            wr_emit<FULL, LUT>(v1, a2, a1, a0, tl, otile + oo, x, W);
            oo += W; ++y;
            a2 = a1; a1 = a0;
#pragma unroll
            for (int k = 0; k < 4; ++k) v1[k] = v0[k];
        }
    }
}
// (two blocks per SM: the look-ahead needs ~120 registers; three blocks with spills measured 45 % slower)
template <bool LISTED, int MINB>
__global__ void __launch_bounds__(TISEG_THREADS, MINB)
k_wsl_remove(Geom g, const int32_t* __restrict__ lab, const unsigned* __restrict__ mask, const int* __restrict__ lut, int KS,
             int32_t* __restrict__ out, bool vec) {
    const int lane = threadIdx.x & 31;
    const int strips = (g.W + 127) >> 7, bands = (g.H + WR_BAND - 1) / WR_BAND;
    const long long wi = (long long)blockIdx.x * TISEG_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    if (wi >= (long long)strips * bands) return;
    const int band = (int)(wi / strips), strip = (int)(wi - (long long)band * strips);
    const int x = strip * 128 + lane * 4, y0 = band * WR_BAND, y1 = min(y0 + WR_BAND, g.H);
    const bool full = vec && strip * 128 + 127 < g.W;          // (warp-uniform)
    FOR_TILES(LISTED, g, n) {
        // (the tile bases are made opaque register pairs: the compiler otherwise re-derives base + n * P + offset in 64-bit
        //  arithmetic at every access of this issue-bound loop; now an access is one IMAD.WIDE)
        const int32_t* tile = lab + (long long)n * g.P;
        int32_t* otile = out + (long long)n * g.P;
        asm volatile("" : "+l"(tile));
        asm volatile("" : "+l"(otile));
        __builtin_assume(__isGlobal(tile));
        __builtin_assume(__isGlobal(otile));
        if (!LISTED) {                                         // the flood output: inside the mask, ids through the table
            const unsigned* mt = mask + (long long)n * g.H * g.SEG;
            const int* tl = lut + (long long)n * KS;
            asm volatile("" : "+l"(mt));
            asm volatile("" : "+l"(tl));
            __builtin_assume(__isGlobal(mt));
            __builtin_assume(__isGlobal(tl));
            if (full) wr_strip<true, true, true>(g, tile, mt, tl, otile, lane, x, y0, y1);
            else wr_strip<false, true, true>(g, tile, mt, tl, otile, lane, x, y0, y1);
        } else {                                               // the general relabelling: a complete map, final ids
            if (full) wr_strip<true, false, false>(g, tile, nullptr, nullptr, otile, lane, x, y0, y1);
            else wr_strip<false, false, false>(g, tile, nullptr, nullptr, otile, lane, x, y0, y1);
        }
    }
}

int h_reconstruction_erosion_dev(tiseg_ctx* c, const Geom& g, const uint8_t* img, int h, uint8_t* out);   // recon.cu

// dist: the distance map, of element type `dtype` (TISEG_DTYPE_*)
int postproc_dist_dev(tiseg_ctx* c, const Geom& g, int dtype, const void* dist, int lamb, int32_t* inst, int32_t* markers_out,
                      int32_t* ws_out) {
    int N = g.N, KS = g.P + 1;
    size_t total = (size_t)N * g.P;
    const size_t nwords = (size_t)N * g.H * g.SEG;
    uint8_t* I0 = ws<uint8_t>(c, total);
    uint8_t* I = I0;
    uint8_t* low = ws<uint8_t>(c, total);
    int* par = ws<int>(c, total);
    int* rank = ws<int>(c, total);
    int* bpar = ws<int>(c, total);
    int* brank = ws<int>(c, total);
    int32_t* wsl = ws_out ? ws_out : ws<int32_t>(c, total);
    int32_t* arranged = ws<int32_t>(c, total);
    int* nmark = ws<int>(c, (size_t)N);
    int* bg = ws<int>(c, (size_t)N);
    int* flagged = ws<int>(c, (size_t)N + 1);
    int* hist = ws<int>(c, (size_t)N * KS);
    int* first = ws<int>(c, (size_t)N * KS);
    int* lut = ws<int>(c, (size_t)N * KS);
    unsigned* fbits = ws<unsigned>(c, nwords);
    unsigned* mbits = ws<unsigned>(c, nwords);           // F plane of the mask b = (I0 < 255)
    unsigned* cbits = ws<unsigned>(c, nwords);
    unsigned* rbits = ws<unsigned>(c, nwords);
    unsigned* bbits = ws<unsigned>(c, nwords);
    unsigned* lbits = ws<unsigned>(c, nwords);
    if (!I0 || !low || !par || !rank || !bpar || !brank || !wsl || !arranged || !nmark || !bg || !flagged || !hist ||
        !first || !lut || !fbits || !mbits || !cbits || !rbits || !bbits || !lbits) return TISEG_ERR_CUDA;
    int* nflagged = flagged + N;
    int* marea = ws<int>(c, 2 * (size_t)N + 2);          // mask pixels per tile; list of the dense tiles + its length
    if (!marea) return TISEG_ERR_CUDA;
    int* dense = marea + N;
    int* ndense = dense + N;
    TISEG_TRY(zero(c, marea, (2 * (size_t)N + 2) * sizeof(int)));

    // the level image, the mask plane, marea and (lambda = 0) the marker candidates in one pass over the distance map
    TISEG_TRY(with_dtype(dtype, [&](auto z) {
        using TI = decltype(z);
        const bool vec = (g.W % 4 == 0) && aligned_x4<TI>(dist) && (((uintptr_t)I0) & 3) == 0;
        if (lamb == 0)
            TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "k_dist_prep"), (k_dist_prep<TI, true>), fr_grid(g), TISEG_THREADS, 0,
                            g, (const TI*)dist, I0, mbits, cbits, bbits, marea, vec);
        else
            TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "k_dist_prep"), (k_dist_prep<TI, false>), fr_grid(g), TISEG_THREADS, 0,
                            g, (const TI*)dist, I0, mbits, (unsigned*)nullptr, (unsigned*)nullptr, marea, vec);
        return TISEG_OK;
    }));
    // Hrecons (dist.py:120): the identity for the lambda = 0.0 the reference hard-codes (dist.py:281); a real
    // H-minima reconstruction otherwise.  Markers and flood levels come from it, the mask b from the image itself.
    if (lamb > 0) {
        I = ws<uint8_t>(c, total);
        if (!I) return TISEG_ERR_CUDA;
        TISEG_TRY(h_reconstruction_erosion_dev(c, g, I0, lamb, I));
        TISEG_LAUNCH(c, k_plateau_bits, fr_grid(g), TISEG_THREADS, 0, g, I, cbits, bbits, (g.W % 4 == 0) && (((uintptr_t)I) & 3) == 0);
    }
    // blobs of the mask b from its bit plane (4-connected); their tables are filled by the seed scatter below
    const BitPlanes mask = {mbits, nullptr, nullptr, nullptr, nullptr};
    BlobInfo b;
    int* seed_blob = ws<int>(c, total);
    unsigned* sbits = ws<unsigned>(c, nwords);
    if (!seed_blob || !sbits) return TISEG_ERR_CUDA;
    TISEG_TRY(blobs_ccl(c, g, mask, bpar, brank, first, b));
    // markers: regional-minimum plateaus (8-connected, equal value) of I below 255, via the candidate pixels
    const dim3 word_grid((unsigned)(((long long)g.H * g.SEG + TISEG_THREADS - 1) / TISEG_THREADS), (unsigned)N);
    const BitPlanes cand = {cbits, nullptr, nullptr, nullptr, nullptr};
    // (a plateau with a pixel that touches an equal-valued non-candidate is not a regional minimum: low[root] = 1, set
    //  inside the labelling from the tile-local roots in shared memory)
    TISEG_TRY(bitccl_build(c, g, cand, 2, par, lbits, rbits, bbits, low));
    TISEG_LAUNCH(c, k_filter_root_bits, word_grid, TISEG_THREADS, 0, g, low, rbits);
    TISEG_TRY(rank_from_bits(c, g, rbits, rank, nmark));
    TISEG_LAUNCH(c, k_init_label_tables, dim3(8, N), 256, 0, hist, first, KS, nmark);      // first[label] = INT_MAX
    // every marker pixel lies inside the mask b = (I < 255), so the markers are the flood's seed map as they are
    // (the flood writes inside the mask only and the passes below read inside it only: the full map is zero-filled just
    //  when the caller asked for it)
    if (ws_out || markers_out) TISEG_TRY(zero(c, wsl, total * sizeof(int32_t)));
    TISEG_LAUNCH(c, k_marker_scatter, word_grid, TISEG_THREADS, 0, g, cbits, par, low, rank, wsl, mask, bpar, brank, b, seed_blob, sbits);
    if (markers_out) TISEG_CHECK(cudaMemcpyAsync(markers_out, wsl, total * sizeof(int32_t), cudaMemcpyDeviceToDevice, c->stream));
    // blobs with one marker label are filled, the others flooded in the (value, age) order
    TISEG_TRY(blobs_boxes_fill(c, g, mask, bpar, brank, b, wsl));
    BlobMember bm;
    bm.par = nullptr; bm.mask_img = I0; bm.seed_blob = seed_blob; bm.seed_bits = sbits;
    bm.mask_bits = mbits; bm.bpar = bpar; bm.brank = brank;
    TISEG_TRY(watershed_u8_masked_dev(c, g, I, bm, b, wsl));
    // arrange_label: the first raster pixel of every flood label came with the fill / the flood's write-back; the
    // background is 0 unless the mask covers more than half of a tile (then the histogram decides, on those tiles only)
    TISEG_TRY(zero(c, nflagged, sizeof(int)));
    TISEG_TRY(zero(c, fbits, (size_t)N * g.H * g.SEG * sizeof(unsigned)));
    TISEG_LAUNCH(c, k_dense_tiles, (N + 255) / 256, 256, 0, marea, N, g.P, bg, dense, ndense);
    Geom gd = listed_geom(g, dense, ndense);
    TISEG_TRY(label_clean_listed(c, g, dense, ndense, mbits, wsl));    // (the histogram reads whole tiles)
    TISEG_LAUNCH(c, k_ws_hist<true>, dim3(quad_grid(g).x, 1), TISEG_THREADS, 0, gd, wsl, hist, first, KS, (g.W % 4 == 0) && aligned16(wsl));
    TISEG_LAUNCH(c, k_pick_bg, N, 256, 0, hist, KS, nmark, g.P, bg, flagged, nflagged, (const int*)dense, (const int*)ndense);
    //   background 0 (every tile but degenerate ones): ids = rank of each region's first pixel; watershed lines
    //   are found on the flood labels themselves (the renumbering is a bijection)
    TISEG_LAUNCH(c, k_first_bits, dim3(8, N), 256, 0, g, first, KS, nmark, fbits);
    TISEG_TRY(rank_from_bits(c, g, fbits, rank, nullptr));
    TISEG_LAUNCH(c, k_arrange_lut, dim3(8, N), 256, 0, g, first, rank, KS, nmark, lut);
    const dim3 px4_grid((unsigned)(((long long)((g.W + 127) / 128) * ((g.H + WR_BAND - 1) / WR_BAND) + TISEG_WARPS_PER_BLOCK - 1) /
                                   TISEG_WARPS_PER_BLOCK), (unsigned)N);
    TISEG_LAUNCH_AS(c, "k_wsl_remove<false>", (k_wsl_remove<false, 2>), px4_grid, TISEG_THREADS, 0, g, wsl, (const unsigned*)mbits, lut, KS, inst,
                 (g.W % 4 == 0) && aligned16(wsl, inst));
    //   any other background: the general relabelling, on the listed tiles only (no blocks do anything otherwise)
    Geom gl = listed_geom(g, flagged, nflagged);
    const unsigned* roots;
    TISEG_TRY(ccl_build(c, gl, ImgEqI32TileBg{wsl, bg}, 2, par, &roots));
    TISEG_TRY(rank_from_bits(c, gl, roots, rank, nullptr));
    TISEG_TRY(apply_rank(c, gl, par, rank, arranged));
    TISEG_LAUNCH_AS(c, "k_wsl_remove<true>", (k_wsl_remove<true, 2>), dim3(px4_grid.x, 1), TISEG_THREADS, 0, gl, arranged, (const unsigned*)nullptr, (const int*)nullptr, 0, inst,
                 (g.W % 4 == 0) && aligned16(arranged, inst));
    return TISEG_OK;
}

}  // namespace tiseg

using namespace tiseg;

extern "C" int tiseg_postproc_dist_lambda_typed(tiseg_ctx* c, int dtype, const void* dist, int N, int H, int W, int lamb,
                                                int32_t* inst_out, int32_t* markers_out, int32_t* ws_out) {
    TISEG_TRY(check_dtype(dtype, "tiseg_postproc_dist_lambda_typed"));
    if (!c || !dist || !inst_out || lamb < 0 || lamb > 255) { set_error("tiseg_postproc_dist_lambda_typed: bad argument (0 <= lambda <= 255)"); return TISEG_ERR_ARG; }
    Call call(c, "tiseg_postproc_dist_lambda_typed", N, H, W);
    const void* d_dist = call.in_bytes(dist, call.total * dtype_bytes(dtype));
    int32_t* d_inst = call.out(inst_out, call.total);
    int32_t* d_mk = call.out(markers_out, call.total);
    int32_t* d_ws = call.out(ws_out, call.total);
    TISEG_TRY(call.status());
    TISEG_TRY(postproc_dist_dev(c, call.g, dtype, d_dist, lamb, d_inst, d_mk, d_ws));
    return call.finish();
}
