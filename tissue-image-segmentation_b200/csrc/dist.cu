// A8 — DIST postprocess: tiseg/models/segmentors/dist.py:275-284 -> dynamic_watershed_alias (:114-129)
// with prepare_prob (:31-40), H_reconstruction_erosion (:43-57; lambda = 0.0 => identity), find_maxima
// (:60-71), arrange_label (:101-111) and generate_wsl (:83-98).
//
//   d  = int32(clip(dist, 0, 255))             (truncation)             k_dist_prep
//   I  = 255 - uint8(d);  b = d > 0.5  <=>  I < 255
//   markers = label(recon_by_erosion(min(255, I+1), I) - I, masked by b)
//           = 8-connected regional-minimum plateaus of I with value < 255, raster ids
//                                                                       plateau CCL + k_plateau_lower + rank
//   ws = watershed(I, markers, mask=b)                                   K6 (bucket flood)
//   arranged = label(ws, background = most frequent value of ws)         k_ws_hist + k_pick_bg + CCL
//   arranged[3x3 window holds >= 2 different non-zero labels] = 0        k_wsl_remove
#include "ccl.cuh"
#include "watershed.cuh"

namespace tiseg {

// level image + the F plane of the mask b = (I < 255): one warp = 128 columns x DP_ROWS rows, four pixels per thread and
// row, all loads of the thread issued before the first is used.  The distance map may be fp32, fp16 or bf16 (TI); it is
// converted to fp32 as it is loaded.
#define DP_ROWS 4
#define PB_ROWS_PER_WARP 32     // rows per warp band of k_plateau_bits (a multiple of 4)
template <bool FULL, class TI>
__device__ __forceinline__ void dp_rows(const Geom& g, const TI* __restrict__ dt, uint8_t* __restrict__ It, unsigned* __restrict__ Ft,
                                        int lane, int x, int y0) {
    const int W = g.W;
    float d[DP_ROWS][4];
#pragma unroll
    for (int r = 0; r < DP_ROWS; ++r) {
        const int y = y0 + r;
        d[r][0] = d[r][1] = d[r][2] = d[r][3] = 0.f;
        if (y < g.H) {                               // (uniform)
            const int ro = y * W + x;
            if (FULL) ld4f_aligned(dt + ro, d[r]);
            else {
#pragma unroll
                for (int k = 0; k < 4; ++k) if (x + k < W) d[r][k] = to_f32(dt[ro + k]);
            }
        }
    }
    const int seg = x >> 5, sh = (lane & 7) * 4;
#pragma unroll
    for (int r = 0; r < DP_ROWS; ++r) {
        const int y = y0 + r;
        if (y >= g.H) break;                         // (uniform)
        const int ro = y * W + x;
        unsigned pack = 0, nib = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float v = d[r][k];
            if (v > 255.f) v = 255.f;      // dist.py:277-278 (comparisons are false for NaN, like numpy)
            if (v < 0.f) v = 0.f;
            const int t = (int)v;          // astype('int32'): truncation
            const unsigned lv = (unsigned)(255 - (t & 255)) & 255u;
            pack |= lv << (8 * k);
            if ((FULL || x + k < W) && lv < 255u) nib |= 1u << k;
        }
        if (FULL) *reinterpret_cast<unsigned*>(It + ro) = pack;
        else {
#pragma unroll
            for (int k = 0; k < 4; ++k) if (x + k < W) It[ro + k] = (uint8_t)(pack >> (8 * k));
        }
        unsigned word = nib << sh;
        word |= __shfl_xor_sync(0xffffffffu, word, 1);
        word |= __shfl_xor_sync(0xffffffffu, word, 2);
        word |= __shfl_xor_sync(0xffffffffu, word, 4);
        if ((lane & 7) == 0 && seg < g.SEG) Ft[y * g.SEG + seg] = word;
    }
}
template <class TI>
__global__ void __launch_bounds__(TISEG_THREADS)
k_dist_prep(Geom g, const TI* __restrict__ dist, uint8_t* __restrict__ I, unsigned* __restrict__ F, bool vec) {
    const int lane = threadIdx.x & 31;
    const int strips = (g.W + 127) >> 7, chunks = (g.H + DP_ROWS - 1) / DP_ROWS;
    const long long wi = (long long)blockIdx.x * TISEG_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    if (wi >= (long long)strips * chunks) return;
    const int ch = (int)(wi / strips), strip = (int)(wi - (long long)ch * strips), n = blockIdx.y;
    // (tile bases as opaque register pairs + 32-bit offsets: one IMAD.WIDE per access)
    const TI* dt = dist + (long long)n * g.P;
    uint8_t* It = I + (long long)n * g.P;
    unsigned* Ft = F + (long long)n * g.H * g.SEG;
    asm volatile("" : "+l"(dt)); asm volatile("" : "+l"(It)); asm volatile("" : "+l"(Ft));
    __builtin_assume(__isGlobal(dt)); __builtin_assume(__isGlobal(It)); __builtin_assume(__isGlobal(Ft));
    if (vec && strip * 128 + 127 < g.W) dp_rows<true>(g, dt, It, Ft, lane, strip * 128 + lane * 4, ch * DP_ROWS);
    else dp_rows<false>(g, dt, It, Ft, lane, strip * 128 + lane * 4, ch * DP_ROWS);
}

// pixels of the mask per tile (decides below whether the flood labels can outnumber the background)
__global__ void __launch_bounds__(TISEG_THREADS) k_mask_area(Geom g, const unsigned* __restrict__ F, int* __restrict__ marea) {
    const long long words = (long long)g.H * g.SEG;
    const int n = blockIdx.y;
    int a = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < words; i += (long long)gridDim.x * blockDim.x)
        a += __popc(F[(long long)n * words + i]);
    a = __reduce_add_sync(0xffffffffu, a);
    if ((threadIdx.x & 31) == 0 && a) atomicAdd(&marea[n], a);
}

// Regional-minimum plateaus without labelling every plateau of the image.  A pixel is a CANDIDATE if its value is
// below 255 and no 8-neighbour is strictly lower.  A plateau P (maximal 8-connected set of equal values) is a regional
// minimum iff all its pixels are candidates.  Label the candidates only (equal value, 8-connected): if P is a
// minimum it comes out as one component, none of whose pixels has an equal-valued non-candidate neighbour; if P is
// not, every candidate component C inside it is a proper subset of the connected P, so some pixel of C touches an
// equal-valued pixel outside C — which must be a non-candidate (a candidate would have joined C).  Hence:
// minimum plateaus = candidate components without an "equal-valued non-candidate neighbour" flag.  On a distance map
// the candidates are the few pixels around each nucleus centre.
__device__ __forceinline__ unsigned ld_u8x4(const uint8_t* __restrict__ row, int x, int W, unsigned oob, bool vec) {
    if (vec) return *reinterpret_cast<const unsigned*>(row + x);
    unsigned r = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) r |= (x + k < W ? (unsigned)row[x + k] : oob) << (8 * k);
    return r;
}
// Candidates are a few percent of the pixels, so the plateau labelling works on one 32-bit word per 32-pixel row
// segment (bits[n, y, seg]) and touches `par` / `low` only at the first pixel of each in-word run of candidates (the
// nodes of the union-find).  Adjacent candidates always carry the same level (the higher one would have a lower
// neighbour), so the labelling is binary.
//   k_plateau_bits         candidate bitmap + bitmap of the candidates that touch an equal-valued non-candidate
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

// Candidate and "bad candidate" bitmaps in one sweep.  With J = I where a pixel is NOT a candidate and 255 where it
// is, a candidate p touches an equal-valued non-candidate iff min3x3(J)(p) == I(p) (every neighbour of a candidate is
// >= it).  So both maps are 3x3 minima.  A thread owns four pixels of a row as two u16x2 words (pixels 0,1 / 2,3) so
// that a three-way minimum of two pixels is ONE instruction (VIMNMX3.U16x2, __vimin3_u16x2); a warp walks down
// PB_ROWS rows of a 32-thread (128-pixel) wide column band keeping the last three row minima in registers, left / right
// pixels come from the neighbouring lanes.  The outer four threads on each side are halo (the stencil of a stencil
// needs two pixels), so a warp emits 24 x 4 pixels = three bitmap words per row.  Lane <-> column mapping: lanes
// 0..23 = output columns, 24..27 = right halo, 28..31 = left halo (neighbours by lane rotation).
struct Px4 { unsigned lo, hi; };                      // (px0 | px1 << 16), (px2 | px3 << 16)
__device__ __forceinline__ Px4 pb_hmin(Px4 v, int lane) {
    const unsigned hl = __shfl_sync(0xffffffffu, v.hi, (lane + 31) & 31);      // pixels 2,3 of the thread to the left
    const unsigned lr = __shfl_sync(0xffffffffu, v.lo, (lane + 1) & 31);       // pixels 0,1 of the thread to the right
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
__global__ void __launch_bounds__(TISEG_THREADS)
k_plateau_bits(Geom g, const uint8_t* __restrict__ I, unsigned* __restrict__ cbits, unsigned* __restrict__ badbits,
               int* __restrict__ par, uint8_t* __restrict__ low, bool vec, int PB_ROWS) {
    const int lane = threadIdx.x & 31;
    const int W4 = (g.W + 3) >> 2, S = (W4 + 23) / 24, bands = (g.H + PB_ROWS - 1) / PB_ROWS;
    const long long wi = (long long)blockIdx.x * TISEG_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    if (wi >= (long long)S * bands) return;
    const int band = (int)(wi / S), st = (int)(wi - (long long)band * S), n = blockIdx.y;
    const int col = lane < 28 ? lane : lane - 32;
    const int x = (st * 24 + col) * 4, y0 = band * PB_ROWS;
    const bool inx = x >= 0 && x < g.W;
    // (tile bases as opaque register pairs + 32-bit offsets: one IMAD.WIDE per access in this issue-bound loop)
    const uint8_t* It = I + (long long)n * g.P;
    unsigned* cb = cbits + (long long)n * g.H * g.SEG;
    unsigned* bb = badbits + (long long)n * g.H * g.SEG;
    int* parn = par + (long long)n * g.P;
    uint8_t* lown = low + (long long)n * g.P;
    asm volatile("" : "+l"(It)); asm volatile("" : "+l"(cb)); asm volatile("" : "+l"(bb)); asm volatile("" : "+l"(parn)); asm volatile("" : "+l"(lown));
    __builtin_assume(__isGlobal(It)); __builtin_assume(__isGlobal(cb)); __builtin_assume(__isGlobal(bb));
    __builtin_assume(__isGlobal(parn)); __builtin_assume(__isGlobal(lown));
    const int seg = st * 3 + (lane >> 3);
    const bool writer = lane < 24 && (lane & 7) == 0 && seg < g.SEG;
    const Px4 FF = {0x00ff00ffu, 0x00ff00ffu};
    Px4 hI1 = FF, hI2 = FF;          // row minima of I, rows r-1 and r-2
    Px4 hJ1 = FF, hJ2 = FF;          // row minima of J, rows r-2 and r-3
    Px4 I1 = FF, I2 = FF;            // I of rows r-1, r-2
    Px4 C2 = {0u, 0u};               // candidate flags (bits 0 / 16) of row r-2
    const int yend = min(y0 + PB_ROWS, g.H);
    for (int r0 = y0 - 2; r0 < yend + 2; r0 += 4) {
        unsigned cw[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {                    // four independent loads in flight
            const int r = r0 + k;
            cw[k] = (inx && r >= 0 && r < g.H) ? ld_u8x4(It + r * g.W, x, g.W, 255u, vec) : 0xffffffffu;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int r = r0 + k;
            Px4 c;
            c.lo = __byte_perm(cw[k], 0u, 0x4140);
            c.hi = __byte_perm(cw[k], 0u, 0x4342);
            const Px4 hI0 = pb_hmin(c, lane);
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
            const Px4 hJ0 = pb_hmin(J, lane);
            // bad candidates of row r-2
            const unsigned jlo = __vimin3_u16x2(hJ0.lo, hJ1.lo, hJ2.lo), jhi = __vimin3_u16x2(hJ0.hi, hJ1.hi, hJ2.hi);
            const unsigned Blo = C2.lo & ~pb_nonzero(jlo ^ I2.lo), Bhi = C2.hi & ~pb_nonzero(jhi ^ I2.hi);
            const int y = r - 2;
            if (y >= y0 && y < yend) {                   // (uniform)
                unsigned w = (pb_nibble(C2.lo, C2.hi) | (pb_nibble(Blo, Bhi) << 16)) << (lane & 3) * 4;
                // eight lanes x four pixels -> one 32-bit word of each map: lanes 0..3 of a group fill the low
                // half-words, lanes 4..7 the high ones
                w |= __shfl_xor_sync(0xffffffffu, w, 1);
                w |= __shfl_xor_sync(0xffffffffu, w, 2);
                const unsigned o = __shfl_xor_sync(0xffffffffu, w, 4);
                if (writer) {
                    const unsigned cwd = (w & 0xffffu) | (o << 16), bwd = (w >> 16) | (o & 0xffff0000u);
                    const int wo = y * g.SEG + seg;
                    cb[wo] = cwd;
                    bb[wo] = bwd;
                    unsigned starts = cwd & ~(cwd << 1);
                    const int idx0 = y * g.W + seg * 32;
                    while (starts) {
                        const int a = __ffs(starts) - 1;
                        starts &= starts - 1;
                        parn[idx0 + a] = idx0 + a;
                        lown[idx0 + a] = 0;
                    }
                }
            }
            hI2 = hI1; hI1 = hI0; hJ2 = hJ1; hJ1 = hJ0; I2 = I1; I1 = c; C2 = C1;
        }
    }
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

    TISEG_TRY(with_dtype(dtype, [&](auto z) {
        using TI = decltype(z);
        const long long warps = (long long)((g.W + 127) / 128) * ((g.H + DP_ROWS - 1) / DP_ROWS);
        TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "k_dist_prep"), k_dist_prep<TI>,
                        dim3((unsigned)((warps + TISEG_WARPS_PER_BLOCK - 1) / TISEG_WARPS_PER_BLOCK), (unsigned)N), TISEG_THREADS, 0,
                        g, (const TI*)dist, I0, mbits, (g.W % 4 == 0) && aligned_x4<TI>(dist) && (((uintptr_t)I0) & 3) == 0);
        return TISEG_OK;
    }));
    // Hrecons (dist.py:120): the identity for the lambda = 0.0 the reference hard-codes (dist.py:281); a real
    // H-minima reconstruction otherwise.  Markers and flood levels come from it, the mask b from the image itself.
    if (lamb > 0) {
        I = ws<uint8_t>(c, total);
        if (!I) return TISEG_ERR_CUDA;
        TISEG_TRY(h_reconstruction_erosion_dev(c, g, I0, lamb, I));
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
    {
        const long long warps = (long long)(((g.W + 3) / 4 + 23) / 24) * ((g.H + PB_ROWS_PER_WARP - 1) / PB_ROWS_PER_WARP);
        TISEG_LAUNCH(c, k_plateau_bits, dim3((unsigned)((warps + TISEG_WARPS_PER_BLOCK - 1) / TISEG_WARPS_PER_BLOCK), (unsigned)N),
                     TISEG_THREADS, 0, g, I, cbits, bbits, par, low, (g.W % 4 == 0) && (((uintptr_t)I) & 3) == 0,
                     PB_ROWS_PER_WARP);
    }
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
    TISEG_LAUNCH(c, k_mask_area, dim3(8, N), TISEG_THREADS, 0, g, mbits, marea);
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
    TISEG_TRY(ccl_build(c, gl, ImgEqI32TileBg{wsl, bg}, 2, par));
    TISEG_TRY(rank_roots(c, gl, par, rank, nullptr));
    TISEG_TRY(apply_rank(c, gl, par, rank, arranged));
    TISEG_LAUNCH_AS(c, "k_wsl_remove<true>", (k_wsl_remove<true, 2>), dim3(px4_grid.x, 1), TISEG_THREADS, 0, gl, arranged, (const unsigned*)nullptr, (const int*)nullptr, 0, inst,
                 (g.W % 4 == 0) && aligned16(arranged, inst));
    return TISEG_OK;
}

}  // namespace tiseg

using namespace tiseg;

extern "C" int tiseg_postproc_dist_lambda(tiseg_ctx* c, const float* dist, int N, int H, int W, int lamb,
                                          int32_t* inst_out, int32_t* markers_out, int32_t* ws_out);

extern "C" int tiseg_postproc_dist(tiseg_ctx* c, const float* dist, int N, int H, int W, int32_t* inst_out,
                                   int32_t* markers_out, int32_t* ws_out) {
    return tiseg_postproc_dist_lambda(c, dist, N, H, W, 0, inst_out, markers_out, ws_out);
}

extern "C" int tiseg_postproc_dist_lambda_typed(tiseg_ctx* c, int dtype, const void* dist, int N, int H, int W, int lamb,
                                                int32_t* inst_out, int32_t* markers_out, int32_t* ws_out) {
    TISEG_TRY(check_dtype(dtype, "tiseg_postproc_dist"));
    if (!c || !dist || !inst_out || lamb < 0 || lamb > 255) { set_error("tiseg_postproc_dist: bad argument (0 <= lambda <= 255)"); return TISEG_ERR_ARG; }
    TISEG_TRY(check_geom(N, H, W));
    begin_call(c);
    Geom g = make_geom(N, H, W);
    size_t total = (size_t)N * g.P;
    const void* d_dist = in_ptr(c, dist, total * dtype_bytes(dtype));
    int32_t* d_inst = tiseg::out(c, inst_out, total);
    int32_t* d_mk = markers_out ? tiseg::out(c, markers_out, total) : nullptr;
    int32_t* d_ws = ws_out ? tiseg::out(c, ws_out, total) : nullptr;
    if (!d_dist || !d_inst) return TISEG_ERR_CUDA;
    TISEG_TRY(postproc_dist_dev(c, g, dtype, d_dist, lamb, d_inst, d_mk, d_ws));
    return end_call(c);
}

extern "C" int tiseg_postproc_dist_lambda(tiseg_ctx* c, const float* dist, int N, int H, int W, int lamb,
                                          int32_t* inst_out, int32_t* markers_out, int32_t* ws_out) {
    return tiseg_postproc_dist_lambda_typed(c, TISEG_DTYPE_F32, dist, N, H, W, lamb, inst_out, markers_out, ws_out);
}
