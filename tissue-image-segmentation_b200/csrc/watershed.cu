// K6 — ordered marker-controlled watershed: blob bookkeeping, the warp-cooperative uint8 flood, the ranked fp64
// bucket flood with its heap fallback, and the tiseg_watershed_* entry points.  See watershed.cuh for the algorithm
// statement.
#include "watershed.cuh"

namespace tiseg {

#define FULL 0xffffffffu

__global__ void k_blob_init(BlobInfo b, int W) {
    int n = blockIdx.y;
    long long o = (long long)n * b.KS;
    int k = b.count[n];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i <= k; i += gridDim.x * blockDim.x) {
        b.root[o + i] = 0; b.ymax[o + i] = -1; b.xmin[o + i] = W; b.xmax[o + i] = -1; b.area[o + i] = 0;
        if (b.lmin) { b.lmin[o + i] = 0x7fffffff; b.lmax[o + i] = 0; }
    }
}

// root[id] = flat index of the blob's first pixel, from the bitmap of the roots (P/32 words instead of the forest)
__global__ void __launch_bounds__(TISEG_THREADS)
k_blob_roots(Geom g, const unsigned* __restrict__ bits, const int* __restrict__ rank, BlobInfo b) {
    const long long words = (long long)g.H * g.SEG;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= words) return;
    const int n = blockIdx.y;
    unsigned m = bits[(long long)n * words + t];
    if (!m) return;
    const int y = (int)(t / g.SEG), seg = (int)(t - (long long)y * g.SEG);
    while (m) {
        const int bit = __ffs(m) - 1;
        m &= m - 1;
        const int idx = y * g.W + seg * 32 + bit;
        b.root[(long long)n * b.KS + rank[(long long)n * g.P + idx]] = idx;
    }
}

// bounding box + area per blob, one set of atomics per in-segment run
__global__ void __launch_bounds__(TISEG_THREADS)
k_blob_bbox(Geom g, const int* __restrict__ par, const int* __restrict__ rank, BlobInfo b, bool vec) {
    Quad q;
    if (!warp_quad(g, q)) return;
    int p[4];
    quad_load_i32(g, q, par + q.base, -1, vec, p);
    if (!__any_sync(FULL, p[0] >= 0 || p[1] >= 0 || p[2] >= 0 || p[3] >= 0)) return;           // (uniform) background only
    const QuadRuns r = quad_runs(p, -1, q.lane);
    FOR_QUAD_RUNS(r, k, len) {
        const long long o = (long long)q.n * b.KS + rank[q.base + p[k]];
        atomicMax(&b.ymax[o], q.y);
        atomicMin(&b.xmin[o], q.x + (int)k);
        atomicMax(&b.xmax[o], q.x + (int)k + (int)len - 1);
        atomicAdd(&b.area[o], (int)len);
    }
}

// off[1..B] = exclusive prefix sum of area[1..B]
__global__ void k_blob_offsets(BlobInfo b) {
    __shared__ int s[256];
    __shared__ int carry;
    int n = blockIdx.x;
    long long o = (long long)n * b.KS;
    int k = b.count[n];
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int base = 1; base <= k; base += 256) {
        int i = base + threadIdx.x;
        int v = i <= k ? b.area[o + i] : 0;
        s[threadIdx.x] = v;
        __syncthreads();
        for (int d = 1; d < 256; d <<= 1) {
            int t = threadIdx.x >= d ? s[threadIdx.x - d] : 0;
            __syncthreads();
            s[threadIdx.x] += t;
            __syncthreads();
        }
        int incl = s[threadIdx.x];
        int c0 = carry;
        if (i <= k) b.off[o + i] = c0 + incl - v;
        __syncthreads();
        if (threadIdx.x == 255) carry = c0 + incl;
        __syncthreads();
    }
}

// ---- blobs from bit planes (DIST) ---------------------------------------------------------------------------------------
// one thread per word of the mask, one step per run piece: the blobs that will be flooded (two or more marker labels)
// collect bounding box + area; the pixels of the others take their label now — the one marker's, or 0 without a marker
// (the label map is not zero-filled, so every mask pixel is written by somebody: here or by the flood).
__global__ void __launch_bounds__(TISEG_THREADS)
k_blob_runs(Geom g, BitPlanes p, const int* __restrict__ par, const int* __restrict__ rank, BlobInfo b, int32_t* __restrict__ out) {
    const long long words = (long long)g.H * g.SEG;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= words) return;
    const int n = blockIdx.y;
    const unsigned F = p.F[(long long)n * words + t];
    if (!F) return;
    const int y = (int)(t / g.SEG), seg = (int)(t - (long long)y * g.SEG);
    for (unsigned m = F & ~(F << 1); m; m &= m - 1) {
        const int a = __ffs(m) - 1;
        const unsigned rest = ~F >> a;                        // (bit 0 is clear: a is in the mask)
        const int len = rest ? __ffs(rest) - 1 : 32 - a;
        const int x = seg * 32 + a;
        const long long o = (long long)n * b.KS + blob_id_at(p, g, n, par, rank, y, x);
        const int lo = b.lmin[o], hi = b.lmax[o];
        if (lo < hi) {
            atomicMax(&b.ymax[o], y);
            atomicMin(&b.xmin[o], x);
            atomicMax(&b.xmax[o], x + len - 1);
            atomicAdd(&b.area[o], len);
        } else {
            const int lab = lo == hi ? lo : 0;
            int32_t* dst = out + (long long)n * g.P + (long long)y * g.W + x;
            for (int k = 0; k < len; ++k) dst[k] = lab;
        }
    }
}
// out = markers * mask (skimage: markers outside the mask are dropped)
__global__ void __launch_bounds__(TISEG_THREADS)
k_ws_seed(long long total, const int32_t* __restrict__ markers, const int* __restrict__ par, int32_t* __restrict__ out, bool vec) {
    const long long i = flat4_index();
    if (i >= total) return;
    Pack4<int> m = ld4(markers, i, total, vec), p = ld4(par, i, total, vec), o;
#pragma unroll
    for (int k = 0; k < 4; ++k) o.v[k] = p.v[k] >= 0 ? m.v[k] : 0;
    st4(out, i, total, vec, o);
}

// ---- work lists and staging, shared by the uint8 and the ranked fp64 flood -----------------------------------------
// A blob's flood is a chain of dependent steps (pop -> look at 4 neighbours -> push), so its speed is the latency
// of the memory it runs in and the number of floods in flight.  Every blob is therefore STAGED into shared memory
// first: the bounding box plus a one-pixel frame (no bounds checks in the flood), flooded there, and written back with
// batched loads/stores.
//
// Both floods (k_ws_flood_par, k_ws_flood_ranked) are persistent kernels (one CTA per SM) fed from work lists sorted by
// size class so that long floods start first.  Framed boxes beyond a warp arena go to a general list, staged by a whole
// CTA: the largest blobs begin at t = 0.  Only boxes beyond that CTA-wide slice are flooded in global memory.
#define WS_NOTIN 0xFFFFu
#define WS_UNLAB 0xFFFEu
#define WS_END 0xFFFFu

#define WS_MAXCLS 16            // most slots per warp arena (= number of size classes)
extern __shared__ __align__(16) unsigned char ws_smem[];

// Work lists of one batch.  An item is (tile << 32) | blob id.  Size class c = blobs whose framed box fits a slot of
// arena / (c + 1) cells but no smaller one, so class 0 holds the largest blobs and is drained first.
struct FloodWork {
    long long* items;   // classes 0..slots-1, contiguous, class c at offset[c] .. offset[c] + count[c]
    long long* gen;     // general list: boxes beyond the warp arena
    long long* ovf;     // ranked flood only: blobs too large to rank or stage, flooded by k_ws_flood_f64
    int* count;         // [WS_MAXCLS]
    int* offset;        // [WS_MAXCLS]
    int* fill;          // [WS_MAXCLS] scatter cursors
    int* cursor;        // [WS_MAXCLS] consumption cursors
    int* ngen;          // [2] lengths of gen, ovf
    int* gcursor;       // [2]
};
#define WK_INTS (4 * WS_MAXCLS + 4)

__device__ __forceinline__ long long blob_cells(const BlobInfo& b, long long ko, int bid, int W) {
    int h = b.ymax[ko + bid] - b.root[ko + bid] / W + 1, w = b.xmax[ko + bid] - b.xmin[ko + bid] + 1;
    return (long long)(w + 2) * (h + 2);
}
__device__ __forceinline__ int blob_class(long long cells, int arena, int slots) {
    if (cells > arena) return -1;
    int cls = arena / (int)cells - 1;
    return cls >= slots ? slots - 1 : cls;
}

// listed tiles (those with a blob beyond `gen_cap` framed cells, flooded in global memory ON the label map): the non-seed
// pixels of exactly those blobs become 0 = "not reached yet"
__global__ void __launch_bounds__(TISEG_THREADS)
k_huge_clean(Geom g, BitPlanes p, const int* __restrict__ par, const int* __restrict__ rank, BlobInfo b,
             const unsigned* __restrict__ seed_bits, long long gen_cap, int32_t* __restrict__ out) {
    const long long words = (long long)g.H * g.SEG;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= words) return;
    const int y = (int)(t / g.SEG), seg = (int)(t - (long long)y * g.SEG);
    FOR_TILES(true, g, n) {
        const unsigned F = p.F[(long long)n * words + t];
        const unsigned seeds = seed_bits[(long long)n * words + t];
        for (unsigned m = F & ~(F << 1); m; m &= m - 1) {
            const int a = __ffs(m) - 1;
            const unsigned rest = ~F >> a;
            const int len = rest ? __ffs(rest) - 1 : 32 - a;
            const int x = seg * 32 + a;
            const long long ko = (long long)n * b.KS;
            const int bid = blob_id_at(p, g, n, par, rank, y, x);
            if (b.lmin[ko + bid] >= b.lmax[ko + bid] || blob_cells(b, ko, bid, g.W) <= gen_cap) continue;
            int32_t* dst = out + (long long)n * g.P + (long long)y * g.W + x;
            for (int k = 0; k < len; ++k) if (!((seeds >> (a + k)) & 1u)) dst[k] = 0;
        }
    }
}

__global__ void k_flood_count(BlobInfo b, int W, FloodWork wk, int arena, int slots) {
    int n = blockIdx.y;
    long long ko = (long long)n * b.KS;
    int B = b.count[n];
    for (int bid = 1 + blockIdx.x * blockDim.x + threadIdx.x; bid <= B; bid += gridDim.x * blockDim.x) {
        if (b.lmin && b.lmin[ko + bid] >= b.lmax[ko + bid]) {
            // a single-marker blob is one region of that label: its first pixel is the blob's
            if (b.first && b.lmax[ko + bid] > 0 && b.lmin[ko + bid] == b.lmax[ko + bid])
                atomicMin(&b.first[ko + b.lmax[ko + bid]], b.root[ko + bid]);
            continue;
        }
        int cls = blob_class(blob_cells(b, ko, bid, W), arena, slots);
        if (cls >= 0) atomicAdd(&wk.count[cls], 1);
    }
}
__global__ void k_flood_offsets(FloodWork wk) {
    if (threadIdx.x == 0) {
        int acc = 0;
        for (int k = 0; k < WS_MAXCLS; ++k) { wk.offset[k] = acc; acc += wk.count[k]; }
    }
}
// `huge` (may be null): [N] flags, [N] list, [1] length — the tiles that hold a blob beyond `gen_cap` cells (those are
// flooded in global memory, on the label map itself, which must then be clean around the seeds: label_clean_listed)
__global__ void k_flood_scatter(BlobInfo b, int W, FloodWork wk, int arena, int slots, long long gen_cap, int* huge) {
    int n = blockIdx.y;
    long long ko = (long long)n * b.KS;
    int B = b.count[n];
    for (int bid = 1 + blockIdx.x * blockDim.x + threadIdx.x; bid <= B; bid += gridDim.x * blockDim.x) {
        if (b.lmin && b.lmin[ko + bid] >= b.lmax[ko + bid]) continue;
        const long long cells = blob_cells(b, ko, bid, W);
        int cls = blob_class(cells, arena, slots);
        long long item = ((long long)n << 32) | (unsigned)bid;
        if (cls >= 0) wk.items[wk.offset[cls] + atomicAdd(&wk.fill[cls], 1)] = item;
        else {
            wk.gen[atomicAdd(wk.ngen, 1)] = item;
            if (huge && cells > gen_cap && atomicExch(&huge[n], 1) == 0) huge[gridDim.y + atomicAdd(&huge[2 * gridDim.y], 1)] = n;
        }
    }
}
// label map of the listed tiles: zero wherever `keep` (a bit plane) is clear
__global__ void __launch_bounds__(TISEG_THREADS)
k_label_clean(Geom g, const unsigned* __restrict__ keep, int32_t* __restrict__ lab) {
    const long long words = (long long)g.H * g.SEG;
    const long long wi = (long long)blockIdx.x * TISEG_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (wi >= words) return;
    const int y = (int)(wi / g.SEG), seg = (int)(wi - (long long)y * g.SEG), x = seg * 32 + lane;
    FOR_TILES(true, g, n) {
        const unsigned w = keep[(long long)n * words + wi];
        if (x < g.W && !((w >> lane) & 1u)) lab[(long long)n * g.P + (long long)y * g.W + x] = 0;
    }
}
int label_clean_listed(tiseg_ctx* c, const Geom& g, const int* list, const int* count, const unsigned* keep, int32_t* lab) {
    Geom gl = listed_geom(g, list, count);
    TISEG_LAUNCH(c, k_label_clean, dim3((unsigned)(((long long)g.H * g.SEG + TISEG_WARPS_PER_BLOCK - 1) / TISEG_WARPS_PER_BLOCK), 1),
                 TISEG_THREADS, 0, gl, keep, lab);
    return TISEG_OK;
}

// floor(j / wp) for j * wp < 2^32 with magic = 0xFFFFFFFF / wp + 1
__device__ __forceinline__ int fdiv(int j, unsigned magic) { return (int)__umulhi((unsigned)j, magic); }

// Per-thread by-products of staging a blob (the caller reduces them if it wants them): the range [lmn, lmx] of the seed
// labels seen and the lowest seed cell — a blob whose seeds all carry ONE label needs no ordered flood at all.
struct SeedStats { int lmn, lmx, jseed; };
// membership of a staged cell (see BlobMember in watershed.cuh)
struct InForest {
    static constexpr bool kMasked = false;
    const int* tp; int root;
    __device__ __forceinline__ int load(int gi) const { return tp[gi]; }
    __device__ __forceinline__ bool in(int v) const { return v == root; }
    // seed <=> the label map holds a label there (ov); the label range of the blob's seeds is a by-product
    __device__ __forceinline__ bool seed(int, unsigned, int, int ov) const { return ov != 0; }
    __device__ __forceinline__ unsigned seed_word(int, int) const { return 0u; }
};
struct InMask {
    static constexpr bool kMasked = true;
    const uint8_t* m; const int* seed_blob; const unsigned* sbits; int SEG; int bid;
    __device__ __forceinline__ int load(int gi) const { return m[gi]; }
    __device__ __forceinline__ bool in(int v) const { return v < 255; }
    __device__ __forceinline__ unsigned seed_word(int y, int x) const { return sbits[y * SEG + (x >> 5)]; }
    __device__ __forceinline__ bool seed(int gi, unsigned word, int x, int) const {
        return ((word >> (x & 31)) & 1u) && seed_blob[gi] == bid;
    }
};

// ---- helpers of the ranked fp64 flood: FIFO buckets, one lane per staged blob -----------------------------------------
// A staged cell takes 4 bytes: the local index of the seed cell whose label it inherits (u16), and one 16-bit field that
// holds the level until the cell is labelled and its FIFO link afterwards (the level is dead by then).
//
// Copy the framed box of a blob into shared memory: lab = own index (seed), UNLAB (in the blob), NOTIN; lvl = level.
// `tid`/`nthr`: the cooperating threads (a warp or a CTA); eight cells per thread are loaded before any is used.
template <class IT, class LT>
__device__ __forceinline__ SeedStats stage_copy(int tid, int nthr, int W, const IT* __restrict__ I, const InForest mb,
                                                const int32_t* __restrict__ o, int root,
                                                int y0, int x0, int w, int h, unsigned short* lab, LT* lvl) {
    SeedStats st; st.lmn = 0x7fffffff; st.lmx = 0; st.jseed = 0x7fffffff;
    const int wp = w + 2, cells = wp * (h + 2);
    const unsigned magic = 0xFFFFFFFFu / (unsigned)wp + 1u;
    for (int j0 = 0; j0 < cells; j0 += 8 * nthr) {
        int gi[8];
        bool in[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int j = j0 + u * nthr + tid;
            const int ly = fdiv(j, magic), lx = j - ly * wp;
            in[u] = j < cells && ly >= 1 && ly <= h && lx >= 1 && lx <= w;
            gi[u] = in[u] ? (y0 + ly - 1) * W + x0 + lx - 1 : root;
        }
        int tpv[8], ov[8];
        IT iv[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) { tpv[u] = mb.load(gi[u]); iv[u] = I[gi[u]]; ov[u] = o[gi[u]]; }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int j = j0 + u * nthr + tid;
            if (j < cells) {
                const bool inblob = in[u] && mb.in(tpv[u]);
                const bool seed = inblob && mb.seed(gi[u], 0u, 0, ov[u]);
                lab[j] = (unsigned short)(inblob ? (seed ? (unsigned)j : WS_UNLAB) : WS_NOTIN);
                lvl[j] = (LT)iv[u];
                if (seed) { st.lmn = min(st.lmn, ov[u]); st.lmx = max(st.lmx, ov[u]); st.jseed = min(st.jseed, j); }
            }
        }
    }
    return st;
}

// warp-level: true if the staged blob has seeds and they all carry one label; then every in-blob cell is pointed at the
// lowest seed cell (the write-back copies that seed's label) and the flood is skipped.  A 4-connected blob is flooded
// completely from any seed, so with a single label there is nothing for the (value, age) order to decide.
__device__ __forceinline__ bool fill_if_single_marker(int lane, SeedStats st, int cells, unsigned short* lab) {
#pragma unroll
    for (int d = 16; d; d >>= 1) {
        st.lmn = min(st.lmn, __shfl_xor_sync(FULL, st.lmn, d));
        st.lmx = max(st.lmx, __shfl_xor_sync(FULL, st.lmx, d));
        st.jseed = min(st.jseed, __shfl_xor_sync(FULL, st.jseed, d));
    }
    if (st.lmx == 0 || st.lmn != st.lmx) return false;
    for (int j = lane; j < cells; j += 32) if (lab[j] == WS_UNLAB) lab[j] = (unsigned short)st.jseed;
    return true;
}

// One warp links the seeds of a staged blob into their buckets in raster order (32 cells per step, the seeds of one
// level inside a step chained with match_any) and returns the level range of the blob and the lowest seed level.
#define WS_LVL_NONE 0x10000        // above every level (uint8 or ranked uint16)
template <class LT, class Bucket>
__device__ __forceinline__ void link_seeds(int lane, int cells, const unsigned short* lab, unsigned short* nxs,
                                           const LT* lvl, unsigned short* head, unsigned short* tail,
                                           Bucket B, int& vmin, int& vmax, int& vsmin) {
    vmin = WS_LVL_NONE; vmax = -1; vsmin = WS_LVL_NONE;
    for (int j0 = 0; j0 < cells; j0 += 32) {
        const int j = j0 + lane;
        unsigned L = WS_NOTIN;
        int v = 0;
        if (j < cells) { L = lab[j]; v = lvl[j]; }
        const bool seed = L == (unsigned)j, inblob = L != WS_NOTIN;
        if (inblob) { vmin = min(vmin, v); vmax = max(vmax, v); }
        if (__ballot_sync(FULL, seed)) {
            const unsigned peers = __match_any_sync(FULL, seed ? v : (WS_LVL_NONE | lane));
            const unsigned below = peers & ((1u << lane) - 1u), above = lane == 31 ? 0u : (peers >> (lane + 1));
            unsigned t = WS_END;
            if (seed) {
                vsmin = min(vsmin, v);
                if (!below) t = tail[B(v)];
            }
            __syncwarp();
            if (seed) {
                nxs[j] = (unsigned short)(above ? (unsigned)(j + __ffs(above)) : WS_END);
                if (!below) { if (t == WS_END) head[B(v)] = (unsigned short)j; else nxs[t] = (unsigned short)j; }
                if (!above) tail[B(v)] = (unsigned short)j;
            }
            __syncwarp();
        }
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) {
        vmin = min(vmin, __shfl_xor_sync(FULL, vmin, d));
        vmax = max(vmax, __shfl_xor_sync(FULL, vmax, d));
        vsmin = min(vsmin, __shfl_xor_sync(FULL, vsmin, d));
    }
}

// The ordered flood of one staged blob by ONE lane (the lanes of a warp flood different slots side by side).  The
// head and tail of the current level's bucket live in registers.  A pop probes the four neighbours' labels; only the
// unlabelled ones (about one per pop on average) run the push body — a loop over the set bits rather than four
// predicated copies, which is what keeps the dependent instruction chain of a step short.
template <class LT, class Bucket>
__device__ __forceinline__ int lane_flood(int wp, int smin, int lmax, unsigned short* lab, unsigned short* nxs,
                                          const LT* lvl, unsigned short* head, unsigned short* tail, Bucket B) {
    int cur = smin, pops = 0;
    unsigned hcur = head[B(cur)], tcur = tail[B(cur)];
    // neighbour offsets up, left, right, down as four signed 16-bit fields
    const unsigned long long offs = ((unsigned long long)(unsigned short)(-wp)) | ((unsigned long long)(unsigned short)(-1) << 16) |
                                    (1ull << 32) | ((unsigned long long)(unsigned short)wp << 48);
    for (;;) {
        if (hcur == WS_END) {
            head[B(cur)] = (unsigned short)WS_END; tail[B(cur)] = (unsigned short)WS_END;
            do { ++cur; } while (cur <= lmax && (hcur = head[B(cur)]) == WS_END);
            if (cur > lmax) break;
            tcur = tail[B(cur)];
        }
        ++pops;
        const int pix = (int)hcur;
        const unsigned l0 = lab[pix - wp], l1 = lab[pix - 1], l2 = lab[pix + 1], l3 = lab[pix + wp];
        const unsigned short L = lab[pix];
        hcur = nxs[pix];
        unsigned m = (l0 == WS_UNLAB ? 1u : 0u) | (l1 == WS_UNLAB ? 2u : 0u) | (l2 == WS_UNLAB ? 4u : 0u) | (l3 == WS_UNLAB ? 8u : 0u);
        int newcur = cur;
        while (m) {
            const int k = __ffs(m) - 1;
            m &= m - 1;
            const int nb = pix + (int)(short)(offs >> (16 * k));
            const int v = lvl[nb];
            lab[nb] = L;                                          // labelled at push time
            nxs[nb] = (unsigned short)WS_END;
            if (v == cur) {
                if (hcur == WS_END) hcur = (unsigned)nb; else nxs[tcur] = (unsigned short)nb;
                tcur = (unsigned)nb;
            } else {
                const unsigned t = tail[B(v)];                    // (sees the push of an earlier neighbour to the same level)
                if (t == WS_END) head[B(v)] = (unsigned short)nb; else nxs[t] = (unsigned short)nb;
                tail[B(v)] = (unsigned short)nb;
                newcur = min(newcur, v);
            }
        }
        if (newcur < cur) {           // a lower level appeared: park the current bucket and descend
            head[B(cur)] = (unsigned short)hcur;
            tail[B(cur)] = (unsigned short)(hcur == WS_END ? WS_END : tcur);
            cur = newcur;
            hcur = head[B(cur)]; tcur = tail[B(cur)];
        }
    }
    return pops;
}

// Every flooded cell takes the marker label of its seed pixel (eight gathers in flight per thread).
__device__ __forceinline__ void stage_writeback(int tid, int nthr, int W, int32_t* o, int y0, int x0, int w, int h,
                                                const unsigned short* lab) {
    const int wp = w + 2, cells = wp * (h + 2), anchor = y0 * W + x0;
    const unsigned magic = 0xFFFFFFFFu / (unsigned)wp + 1u;
    for (int j0 = 0; j0 < cells; j0 += 8 * nthr) {
        int dst[8], src[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int j = j0 + u * nthr + tid;
            dst[u] = -1; src[u] = anchor;
            if (j < cells) {
                const unsigned L = lab[j];
                if (L < WS_UNLAB && L != (unsigned)j) {
                    const int ly = fdiv(j, magic), lx = j - ly * wp, sy = fdiv((int)L, magic), sx = (int)L - sy * wp;
                    dst[u] = (y0 + ly - 1) * W + x0 + lx - 1;
                    src[u] = (y0 + sy - 1) * W + x0 + sx - 1;
                }
            }
        }
        int val[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) val[u] = o[src[u]];
#pragma unroll
        for (int u = 0; u < 8; ++u) if (dst[u] >= 0) o[dst[u]] = val[u];
    }
}

// The sequential uint8 flood of one blob in global memory, by one lane (framed bounding box too large for shared
// memory): 256 FIFO buckets, head/tail are int[256], the links live in `nx`.
template <class MB>
__device__ __forceinline__ void flood_blob_global(int lane, int W, int H, const uint8_t* __restrict__ I,
                                                  const MB mb, int32_t* o, int* nx, int root, int y0,
                                                  int y1, int x0, int x1, int* head, int* tail, int* first = nullptr) {
    for (int i = lane; i < 256; i += 32) { head[i] = -1; tail[i] = -1; }
    __syncwarp();
    int cur = 256;
    for (int y = y0; y <= y1; ++y) {
        for (int xb = x0; xb <= x1; xb += 32) {
            int x = xb + lane;
            bool seed = false;
            int lv = 0;
            if (x <= x1) {
                int idx = y * W + x;
                if (mb.in(mb.load(idx)) && mb.seed(idx, MB::kMasked ? mb.seed_word(y, x) : 0u, x, o[idx])) { seed = true; lv = I[idx]; }
            }
            unsigned m = __ballot_sync(FULL, seed);
            while (m) {
                int src = __ffs(m) - 1;
                m &= m - 1;
                int slv = __shfl_sync(FULL, lv, src);
                if (lane == 0) {
                    int pix = y * W + xb + src;
                    if (first) atomicMin(&first[o[pix]], pix);
                    nx[pix] = -1;
                    int t = tail[slv];
                    if (t < 0) head[slv] = pix; else nx[t] = pix;
                    tail[slv] = pix;
                    if (slv < cur) cur = slv;
                }
            }
        }
    }
    if (lane == 0) {
        for (;;) {
            while (cur < 256 && head[cur] < 0) ++cur;
            if (cur >= 256) break;
            const int pix = head[cur];
            const int nxt = nx[pix];
            head[cur] = nxt;
            if (nxt < 0) tail[cur] = -1;
            const int lab_g = o[pix];
            const int y = pix / W, x = pix - y * W;
            const int nb[4] = {pix - W, pix - 1, pix + 1, pix + W};
            const bool ok[4] = {y > 0, x > 0, x + 1 < W, y + 1 < H};
            int ov[4], lv[4];
            bool pin[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                pin[k] = false; ov[k] = 1; lv[k] = 0;
                if (ok[k]) { pin[k] = mb.in(mb.load(nb[k])); ov[k] = o[nb[k]]; lv[k] = I[nb[k]]; }
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (pin[k] && ov[k] == 0) {
                    o[nb[k]] = lab_g;
                    if (first) atomicMin(&first[lab_g], nb[k]);
                    nx[nb[k]] = -1;
                    int t = tail[lv[k]];
                    if (t < 0) head[lv[k]] = nb[k]; else nx[t] = nb[k];
                    tail[lv[k]] = nb[k];
                    if (lv[k] < cur) cur = lv[k];
                }
            }
        }
    }
    __syncwarp();
}

// ---- uint8 levels, warp-cooperative flood ---------------------------------------------------------------------------------
// A flood by one lane (as in lane_flood) advances one pixel per ~500 cycles and blob, so a cluster of touching nuclei (a
// blob of 2-3 thousand pixels) alone would last as long as the whole kernel (profiles/r2_flood_debug.txt: mean 0.73 M
// cycles per warp, max 1.04 M).  Here ONE WARP floods one blob and pops up to 32 pixels of the current level per step,
// with exactly the sequential result:
//   * queues are ARRAYS: every cell is pushed at most once, so level v never receives more entries than the blob has
//     cells of level v; the staging pass counts them and the queue storage is cut into one segment per level.  The
//     first B <= 32 entries e_0 .. e_{B-1} of the current level are read by lanes 0 .. B-1.
//   * a cell is packed into one 32-bit word, state << 16 | level (state: NOTIN, UNLAB or the cell index of the seed whose
//     label it inherits).  Lane i claims each unlabelled neighbour k with atomicMin(cell, (4 i + k) << 16 | level): the
//     sequential flood would have given the cell to the first entry in queue order, and to its first neighbour slot, that
//     reaches it — the smallest key.  After a warp barrier the winners are the claims that read their own key back.
//   * pushes enter the queue of their level in (i, k) order: per target level a ballot prefix gives every winner its slot.
//   * if a winner's cell lies BELOW the current level, the sequential flood leaves the current level right after that
//     entry: the step is cut after the first such lane i* (lanes above it put their claims back and stay in the queue),
//     and the flood continues at the lowest new level.
// Cost per step ~ a few hundred cycles whether 1 or 32 pixels are popped, so long queues (big blobs) run ~20x faster and
// short ones no slower.
// Every phase of a blob (staging, queue set-up, flood steps, write-back) is a chain of memory latencies, so the SM wants
// as many blobs in flight as shared memory allows: 4 warps own a big arena (the largest size classes), 12 warps a small
// one (a third of it: size classes >= 2, most blobs).
#define WP_WARPS 16
#define WP_BIG_WARPS 4
#define WP_ARENA 4224                                   // cells of a big warp arena (4 B cell + 2 B queue slot)
#define WP_SMALL_ARENA (WP_ARENA / 3)                   // cells of a small one: size classes >= 2
#define WP_SMALL_CLS 2
#define WP_META_BYTES (256 * 2 * 2 + 128 * 4)           // head, tail (u16 x 256 each), level counts (u16 x 256)
#define WP_GEN_CAP (WP_ARENA * WP_BIG_WARPS + WP_SMALL_ARENA * (WP_WARPS - WP_BIG_WARPS))     // cells of the CTA-wide slice
#define WP_SMEM_BYTES ((size_t)WP_GEN_CAP * 6 + (size_t)WP_META_BYTES * WP_WARPS)
#define WPC_NOTIN 0xFFFFu
#define WPC_UNLAB 0xFFFEu

template <class MB>
__device__ __forceinline__ SeedStats wp_stage(int tid, int nthr, int W, const uint8_t* __restrict__ I, const MB mb,
                                              const int32_t* __restrict__ o, int root, int y0, int x0, int w, int h,
                                              unsigned* cell, unsigned* cnt32) {
    SeedStats st; st.lmn = 0x7fffffff; st.lmx = 0; st.jseed = 0x7fffffff;
    const int wp = w + 2, cells = wp * (h + 2);
    const unsigned magic = 0xFFFFFFFFu / (unsigned)wp + 1u;
    for (int j0 = 0; j0 < cells; j0 += 8 * nthr) {
        int gi[8], gy[8], gx[8];
        bool in[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int j = j0 + u * nthr + tid;
            const int ly = fdiv(j, magic), lx = j - ly * wp;
            in[u] = j < cells && ly >= 1 && ly <= h && lx >= 1 && lx <= w;
            gy[u] = y0 + ly - 1; gx[u] = x0 + lx - 1;
            gi[u] = in[u] ? gy[u] * W + gx[u] : root;
        }
        int mv[8], ov[8];
        unsigned iv[8], sw[8];
        // (all loads of the eight cells in flight together; the seed bitmap word instead of the label map in mask mode)
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            mv[u] = mb.load(gi[u]); iv[u] = I[gi[u]]; ov[u] = MB::kMasked ? 0 : o[gi[u]];
            sw[u] = (MB::kMasked && in[u]) ? mb.seed_word(gy[u], gx[u]) : 0u;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int j = j0 + u * nthr + tid;
            if (j < cells) {
                const bool inblob = in[u] && mb.in(mv[u]);
                const bool seed = inblob && mb.seed(gi[u], sw[u], gx[u], ov[u]);
                cell[j] = ((inblob ? (seed ? (unsigned)j : WPC_UNLAB) : WPC_NOTIN) << 16) | iv[u];
                if (inblob) atomicAdd(&cnt32[iv[u] >> 1], 1u << (16 * (iv[u] & 1u)));
                if (seed) { st.lmn = min(st.lmn, ov[u]); st.lmx = max(st.lmx, ov[u]); st.jseed = min(st.jseed, j); }
            }
        }
    }
    return st;
}

// one warp: queue segments from the level counts, then the seeds in raster order.  Returns the lowest seed level (256 if
// the blob has no seed).
__device__ __forceinline__ int wp_prepare(int lane, int cells, const unsigned* cell, unsigned short* Q, unsigned short* head,
                                          unsigned short* tail, const unsigned* cnt32) {
    // exclusive prefix of the 256 counts: lane l owns levels 8 l .. 8 l + 7
    int c[8], tot = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const unsigned t = cnt32[lane * 4 + k];
        c[2 * k] = (int)(t & 0xffffu); c[2 * k + 1] = (int)(t >> 16);
        tot += c[2 * k] + c[2 * k + 1];
    }
    int incl = tot;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const int t = __shfl_up_sync(FULL, incl, d); if (lane >= d) incl += t; }
    int off = incl - tot;
#pragma unroll
    for (int k = 0; k < 8; ++k) { head[lane * 8 + k] = (unsigned short)off; tail[lane * 8 + k] = (unsigned short)off; off += c[k]; }
    __syncwarp();
    int smin = 256;
    for (int j0 = 0; j0 < cells; j0 += 32) {
        const int j = j0 + lane;
        const unsigned cw = j < cells ? cell[j] : (WPC_NOTIN << 16);
        const bool seed = (cw >> 16) == (unsigned)j;
        if (!__ballot_sync(FULL, seed)) continue;
        const int v = (int)(cw & 0xffffu);
        const unsigned peers = __match_any_sync(FULL, seed ? v : (0x100 | lane));
        if (seed) {
            const int leader = __ffs(peers) - 1;
            const int rank = __popc(peers & ((1u << lane) - 1u));
            const int t = tail[v];                                   // (every peer reads the same value)
            Q[t + rank] = (unsigned short)j;
            smin = min(smin, v);
            __syncwarp(peers);
            if (lane == leader) tail[v] = (unsigned short)(t + __popc(peers));
        }
        __syncwarp();
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) smin = min(smin, __shfl_xor_sync(FULL, smin, d));
    return smin;
}

__device__ __forceinline__ void wp_flood(int lane, int wp, unsigned* cell, unsigned short* Q, unsigned short* head,
                                         unsigned short* tail, int cur) {
    const int offs[4] = {-wp, -1, 1, wp};
    for (;;) {
        const int h = head[cur], t = tail[cur];
        if (h == t) {                                   // next non-empty level (uniform)
            int nxt = -1;
            for (int base = cur + 1; base < 256 && nxt < 0; base += 32) {
                const int l = base + lane;
                const unsigned m = __ballot_sync(FULL, l < 256 && head[l] != tail[l]);
                if (m) nxt = base + __ffs(m) - 1;
            }
            if (nxt < 0) return;
            cur = nxt;
            continue;
        }
        const int B = min(t - h, 32);
        const bool act = lane < B;
        const int e = act ? (int)Q[h + lane] : 0;
        const unsigned L = act ? cell[e] >> 16 : 0u;
        unsigned ck[4];
        bool want[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            ck[k] = act ? cell[e + offs[k]] : (WPC_NOTIN << 16);
            want[k] = (ck[k] >> 16) == WPC_UNLAB;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (want[k]) atomicMin(&cell[e + offs[k]], ((unsigned)(lane * 4 + k) << 16) | (ck[k] & 0xffffu));
        __syncwarp();
        unsigned won = 0;
        bool desc = false;
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (want[k] && (cell[e + offs[k]] >> 16) == (unsigned)(lane * 4 + k)) {
                won |= 1u << k;
                desc |= (int)(ck[k] & 0xffffu) < cur;
            }
        const unsigned dm = __ballot_sync(FULL, desc);
        const int istar = dm ? __ffs(dm) - 1 : B - 1;       // the step ends after the first entry that opens a lower level
        __syncwarp();                                       // every key has been read back before a label replaces one
        const bool keep = lane <= istar;
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if ((won >> k) & 1u) cell[e + offs[k]] = ((keep ? L : WPC_UNLAB) << 16) | (ck[k] & 0xffffu);
        unsigned pend = keep ? won : 0u;
        int newcur = cur;
        for (;;) {
            const unsigned anyp = __ballot_sync(FULL, pend != 0u);
            if (!anyp) break;
            const int k0 = __ffs(pend) - 1;                  // (pend == 0: unused)
            const int myv = pend ? (int)((k0 == 0 ? ck[0] : k0 == 1 ? ck[1] : k0 == 2 ? ck[2] : ck[3]) & 0xffffu) : 0;
            const int v = __shfl_sync(FULL, myv, __ffs(anyp) - 1);
            unsigned mine = 0;
#pragma unroll
            for (int k = 0; k < 4; ++k) if (((pend >> k) & 1u) && (int)(ck[k] & 0xffffu) == v) mine |= 1u << k;
            const unsigned b0 = __ballot_sync(FULL, mine & 1u), b1 = __ballot_sync(FULL, mine & 2u);
            const unsigned b2 = __ballot_sync(FULL, mine & 4u), b3 = __ballot_sync(FULL, mine & 8u);
            const unsigned below = (1u << lane) - 1u;
            const int pre = __popc(b0 & below) + __popc(b1 & below) + __popc(b2 & below) + __popc(b3 & below);
            const int tot = __popc(b0) + __popc(b1) + __popc(b2) + __popc(b3);
            const int tv = tail[v];
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if ((mine >> k) & 1u) Q[tv + pre + __popc(mine & ((1u << k) - 1u))] = (unsigned short)(e + offs[k]);
            __syncwarp();
            if (lane == 0) tail[v] = (unsigned short)(tv + tot);
            pend &= ~mine;
            newcur = min(newcur, v);
            __syncwarp();
        }
        if (lane == 0) head[cur] = (unsigned short)(h + istar + 1);
        __syncwarp();
        cur = newcur;
    }
}

// every labelled cell takes the marker label of its seed pixel; `first` (may be NULL): lowest flat index per label, one
// atomic per run of equal labels along the staged rows
__device__ __forceinline__ void wp_writeback(int tid, int nthr, int W, int32_t* o, int y0, int x0, int w, int h, const unsigned* cell,
                                             int* first) {
    const int wp = w + 2, cells = wp * (h + 2), anchor = y0 * W + x0;
    const unsigned magic = 0xFFFFFFFFu / (unsigned)wp + 1u;
    for (int j0 = 0; j0 < cells; j0 += 8 * nthr) {
        int dst[8], src[8];
        bool store[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int j = j0 + u * nthr + tid;
            dst[u] = -1; src[u] = anchor; store[u] = false;
            if (j < cells) {
                const unsigned L = cell[j] >> 16;
                if (L < WPC_UNLAB) {
                    const int ly = fdiv(j, magic), lx = j - ly * wp, sy = fdiv((int)L, magic), sx = (int)L - sy * wp;
                    dst[u] = (y0 + ly - 1) * W + x0 + lx - 1;
                    src[u] = (y0 + sy - 1) * W + x0 + sx - 1;
                    store[u] = L != (unsigned)j;
                }
            }
        }
        int val[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) val[u] = o[src[u]];
#pragma unroll
        for (int u = 0; u < 8; ++u) if (store[u]) o[dst[u]] = val[u];
        if (first) {
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int key = dst[u] >= 0 ? val[u] : 0;
                const int left = __shfl_up_sync(FULL, key, 1);
                if (key != 0 && ((tid & 31) == 0 || left != key)) atomicMin(&first[key], dst[u]);
            }
        }
    }
}

template <bool MASKED>
__global__ void __launch_bounds__(32 * WP_WARPS, 1)
k_ws_flood_par(Geom g, const uint8_t* __restrict__ image, BlobMember bm, BlobInfo b, FloodWork wk, int* next, int* gheads,
               int32_t* out) {
    __shared__ int s_item;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int W = g.W, H = g.H;
    // ---- blobs beyond one warp arena: the whole CTA stages, one warp floods (largest first: they start at t = 0)
    {
        unsigned* cell = reinterpret_cast<unsigned*>(ws_smem);
        unsigned short* Q = reinterpret_cast<unsigned short*>(cell + WP_GEN_CAP);
        unsigned short* head = reinterpret_cast<unsigned short*>(ws_smem + (size_t)WP_GEN_CAP * 6);
        unsigned short* tail = head + 256;
        unsigned* cnt32 = reinterpret_cast<unsigned*>(tail + 256);
        const int ngen = wk.ngen[0];
        for (;;) {
            __syncthreads();
            if (threadIdx.x == 0) s_item = atomicAdd(wk.gcursor, 1);
            __syncthreads();
            const int k = s_item;
            if (k >= ngen) break;
            const long long item = wk.gen[k];
            const int n = (int)(item >> 32), bid = (int)(item & 0xffffffffll);
            const long long base = (long long)n * g.P, ko = (long long)n * b.KS;
            const int root = b.root[ko + bid];
            const int y0 = root / W, y1 = b.ymax[ko + bid], x0 = b.xmin[ko + bid], x1 = b.xmax[ko + bid];
            const int w = x1 - x0 + 1, h = y1 - y0 + 1;
            const long long cells = (long long)(w + 2) * (h + 2);
            const InForest inf = {bm.par + base, root};
            const InMask inm = {MASKED ? bm.mask_img + base : nullptr, MASKED ? bm.seed_blob + base : nullptr,
                                MASKED ? bm.seed_bits + (long long)n * g.H * g.SEG : nullptr, g.SEG, bid};
            if (cells > WP_GEN_CAP) {     // does not fit: the sequential flood in global memory, by one lane
                if (warp == 0) {
                    int* fst = b.first ? b.first + ko : nullptr;
                    if (MASKED) flood_blob_global(lane, W, H, image + base, inm, out + base, next + base, root, y0, y1, x0, x1,
                                                  gheads + (size_t)blockIdx.x * 512, gheads + (size_t)blockIdx.x * 512 + 256, fst);
                    else flood_blob_global(lane, W, H, image + base, inf, out + base, next + base, root, y0, y1, x0, x1,
                                           gheads + (size_t)blockIdx.x * 512, gheads + (size_t)blockIdx.x * 512 + 256, fst);
                }
                continue;
            }
            for (int i = threadIdx.x; i < 128; i += blockDim.x) cnt32[i] = 0u;
            __syncthreads();
            if (MASKED) wp_stage(threadIdx.x, blockDim.x, W, image + base, inm, out + base, root, y0, x0, w, h, cell, cnt32);
            else wp_stage(threadIdx.x, blockDim.x, W, image + base, inf, out + base, root, y0, x0, w, h, cell, cnt32);
            __syncthreads();
            if (warp == 0) {
                const int smin = wp_prepare(lane, (int)cells, cell, Q, head, tail, cnt32);
                if (smin < 256) wp_flood(lane, w + 2, cell, Q, head, tail, smin);
            }
            __syncthreads();
            wp_writeback(threadIdx.x, blockDim.x, W, out + base, y0, x0, w, h, cell, b.first ? b.first + ko : nullptr);
        }
        __syncthreads();
    }
    // ---- one blob per warp, size classes from the largest to the smallest
    const bool big = warp < WP_BIG_WARPS;
    const int arena = big ? WP_ARENA : WP_SMALL_ARENA;
    unsigned char* wbase = ws_smem + (big ? (size_t)warp * WP_ARENA * 6
                                          : (size_t)WP_BIG_WARPS * WP_ARENA * 6 + (size_t)(warp - WP_BIG_WARPS) * WP_SMALL_ARENA * 6);
    unsigned* cell = reinterpret_cast<unsigned*>(wbase);
    unsigned short* Q = reinterpret_cast<unsigned short*>(cell + arena);
    unsigned short* head = reinterpret_cast<unsigned short*>(ws_smem + (size_t)WP_GEN_CAP * 6 + (size_t)warp * WP_META_BYTES);
    unsigned short* tail = head + 256;
    unsigned* cnt32 = reinterpret_cast<unsigned*>(tail + 256);
    for (int cls = big ? 0 : WP_SMALL_CLS; cls < WS_MAXCLS; ++cls) {
        const int cnt = wk.count[cls];
        const long long* list = wk.items + wk.offset[cls];
        for (;;) {
            int k = 0;
            if (lane == 0) k = atomicAdd(&wk.cursor[cls], 1);
            k = __shfl_sync(FULL, k, 0);
            if (k >= cnt) break;
            const long long item = list[k];
            const int n = (int)(item >> 32), bid = (int)(item & 0xffffffffll);
            const long long base = (long long)n * g.P, ko = (long long)n * b.KS;
            const int root = b.root[ko + bid];
            const int y0 = root / W, x0 = b.xmin[ko + bid];
            const int w = b.xmax[ko + bid] - x0 + 1, h = b.ymax[ko + bid] - y0 + 1;
            const int cells = (w + 2) * (h + 2);
            for (int i = lane; i < 128; i += 32) cnt32[i] = 0u;
            __syncwarp();
            bool flood = true;
            if (MASKED) {
                const InMask inm = {bm.mask_img + base, bm.seed_blob + base, bm.seed_bits + (long long)n * g.H * g.SEG, g.SEG, bid};
                wp_stage(lane, 32, W, image + base, inm, out + base, root, y0, x0, w, h, cell, cnt32);
            } else {
                const InForest inf = {bm.par + base, root};
                SeedStats st = wp_stage(lane, 32, W, image + base, inf, out + base, root, y0, x0, w, h, cell, cnt32);
                // all seeds carry one label: a 4-connected blob is flooded completely from any seed, nothing to order
#pragma unroll
                for (int d = 16; d; d >>= 1) {
                    st.lmn = min(st.lmn, __shfl_xor_sync(FULL, st.lmn, d));
                    st.lmx = max(st.lmx, __shfl_xor_sync(FULL, st.lmx, d));
                    st.jseed = min(st.jseed, __shfl_xor_sync(FULL, st.jseed, d));
                }
                __syncwarp();
                if (st.lmx != 0 && st.lmn == st.lmx) {
                    for (int j = lane; j < cells; j += 32)
                        if ((cell[j] >> 16) == WPC_UNLAB) cell[j] = ((unsigned)st.jseed << 16) | (cell[j] & 0xffffu);
                    flood = false;
                }
            }
            __syncwarp();
            if (flood) {
                const int smin = wp_prepare(lane, cells, cell, Q, head, tail, cnt32);
                if (smin < 256) wp_flood(lane, w + 2, cell, Q, head, tail, smin);
            }
            __syncwarp();
            wp_writeback(lane, 32, W, out + base, y0, x0, w, h, cell, b.first ? b.first + ko : nullptr);
            __syncwarp();
        }
    }
}

// ---- fp64 values, fast path: per-blob dense ranks + a bucket flood in shared memory ------------------------------------
// The (value, age) order of the flood only compares values INSIDE one blob, so the fp64 image can be replaced, blob
// by blob, by the dense rank of each pixel's value among the blob's distinct values (equal doubles -> equal rank):
// the flood then runs on small integers with FIFO buckets in shared memory (stage_copy .. stage_writeback), instead of
// a binary heap in global memory.  Ranking = one bitonic sort of the blob's values in shared memory (k_rank_blobs),
// a flag-and-scan for the distinct values, and a binary search per pixel.  Blobs whose framed box exceeds WR_GEN_CAP
// cells or whose area exceeds WR_SORT_MAX keep the heap flood (k_ws_flood_f64).
#define WR_SORT_SMALL 1024        // values sorted by a 128-thread CTA
#define WR_SORT_MAX 16384         // values sorted by a 1024-thread CTA
#define WR_GEN_CAP 28160          // cells of the single-blob slice of the ranked general path (8 B per cell)

__device__ __forceinline__ bool blob_is_huge(const BlobInfo& b, long long ko, int bid, int W) {
    return blob_cells(b, ko, bid, W) > WR_GEN_CAP || b.area[ko + bid] > WR_SORT_MAX;
}

// blob index -> (tile, id): prefix[n] = blobs in the tiles before n (prefix[N] = total)
__global__ void k_blob_prefix(const int* __restrict__ count, int N, int* prefix) {
    if (threadIdx.x == 0) {
        int acc = 0;
        for (int n = 0; n < N; ++n) { prefix[n] = acc; acc += count[n]; }
        prefix[N] = acc;
    }
}

// One CTA per blob (persistent over all blobs of the batch); LARGE = false takes areas <= WR_SORT_SMALL, true the rest
// up to WR_SORT_MAX.  level[pixel] = dense rank of image[pixel] among the blob's values.
template <bool LARGE>
__global__ void __launch_bounds__(LARGE ? 1024 : 128)
k_rank_blobs(Geom g, const double* __restrict__ image, const int* __restrict__ par, BlobInfo b, const int* __restrict__ prefix,
             unsigned short* __restrict__ level) {
    extern __shared__ __align__(16) unsigned char rk_smem[];
    constexpr int CAP = LARGE ? WR_SORT_MAX : WR_SORT_SMALL;
    double* val = reinterpret_cast<double*>(rk_smem);                    // [CAP] sorted values
    unsigned short* rnk = reinterpret_cast<unsigned short*>(val + CAP);  // [CAP] dense rank of sorted position
    __shared__ int s_cnt, s_carry;
    const int N = g.N, W = g.W, total = prefix[N];
    for (int bi = blockIdx.x; bi < total; bi += gridDim.x) {
        int n = 0;                                         // tile of blob bi (N is small: linear search)
        while (n + 1 < N && prefix[n + 1] <= bi) ++n;
        const int bid = bi - prefix[n] + 1;
        const long long ko = (long long)n * b.KS, base = (long long)n * g.P;
        const int area = b.area[ko + bid];
        if (LARGE ? (area <= WR_SORT_SMALL || blob_is_huge(b, ko, bid, W)) : (area > WR_SORT_SMALL)) continue;   // uniform
        const int root = b.root[ko + bid];
        const int y0 = root / W, x0 = b.xmin[ko + bid], w = b.xmax[ko + bid] - x0 + 1, h = b.ymax[ko + bid] - y0 + 1;
        const int box = w * h;
        const unsigned magic = 0xFFFFFFFFu / (unsigned)w + 1u;
        __syncthreads();
        if (threadIdx.x == 0) s_cnt = 0;
        __syncthreads();
        // gather the blob's values (order irrelevant)
        for (int j = threadIdx.x; j < box; j += blockDim.x) {
            const int ly = fdiv(j, magic), lx = j - ly * w;
            const int gi = (y0 + ly) * W + x0 + lx;
            if (par[base + gi] == root) val[atomicAdd(&s_cnt, 1)] = image[base + gi];
        }
        __syncthreads();
        const int cnt = s_cnt;                             // == area
        int n2 = 1;
        while (n2 < cnt) n2 <<= 1;
        for (int j = cnt + threadIdx.x; j < n2; j += blockDim.x) val[j] = INFINITY;
        __syncthreads();
        // bitonic sort, ascending
        for (int k = 2; k <= n2; k <<= 1) {
            for (int d = k >> 1; d > 0; d >>= 1) {
                for (int i = threadIdx.x; i < n2; i += blockDim.x) {
                    const int ixj = i ^ d;
                    if (ixj > i) {
                        const double a = val[i], c = val[ixj];
                        const bool up = (i & k) == 0;
                        if ((a > c) == up) { val[i] = c; val[ixj] = a; }
                    }
                }
                __syncthreads();
            }
        }
        // dense ranks of the sorted positions: inclusive scan of "differs from the previous value", chunk by chunk
        if (threadIdx.x == 0) s_carry = 0;
        __syncthreads();
        for (int c0 = 0; c0 < cnt; c0 += blockDim.x) {
            const int i = c0 + threadIdx.x;
            const int f = (i < cnt && i > 0 && val[i] != val[i - 1]) ? 1 : 0;
            // block inclusive scan of f (warp scans + warp totals in rnk scratch beyond cnt is unsafe: use shuffles + smem)
            int incl = f;
            const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
            for (int dd = 1; dd < 32; dd <<= 1) { int t = __shfl_up_sync(FULL, incl, dd); if (lane >= dd) incl += t; }
            __shared__ int wtot[32];
            if (lane == 31) wtot[wid] = incl;
            __syncthreads();
            if (wid == 0) {
                int wv = lane < (int)(blockDim.x >> 5) ? wtot[lane] : 0, wi = wv;
#pragma unroll
                for (int dd = 1; dd < 32; dd <<= 1) { int t = __shfl_up_sync(FULL, wi, dd); if (lane >= dd) wi += t; }
                wtot[lane] = wi - wv;
            }
            __syncthreads();
            const int r = s_carry + wtot[wid] + incl;
            if (i < cnt) rnk[i] = (unsigned short)r;
            __syncthreads();
            if (threadIdx.x == blockDim.x - 1) s_carry = r;
            __syncthreads();
        }
        // every pixel: first sorted position holding its value -> rank
        for (int j = threadIdx.x; j < box; j += blockDim.x) {
            const int ly = fdiv(j, magic), lx = j - ly * w;
            const int gi = (y0 + ly) * W + x0 + lx;
            if (par[base + gi] != root) continue;
            const double v = image[base + gi];
            int lo = 0, hi = cnt - 1;
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (val[mid] < v) lo = mid + 1; else hi = mid; }
            level[base + gi] = rnk[lo];
        }
    }
}

struct BucketDirect {           // ranked levels index their bucket directly inside the slot's range
    int base;
    __device__ __forceinline__ int operator()(int v) const { return base + v; }
};

// work lists for the ranked flood: like k_flood_count / k_flood_scatter, but huge blobs go to the heap list (ovf)
__global__ void k_flood_count_ranked(BlobInfo b, int W, FloodWork wk, int arena, int slots) {
    int n = blockIdx.y;
    long long ko = (long long)n * b.KS;
    int B = b.count[n];
    for (int bid = 1 + blockIdx.x * blockDim.x + threadIdx.x; bid <= B; bid += gridDim.x * blockDim.x) {
        if (blob_is_huge(b, ko, bid, W)) continue;
        int cls = blob_class(blob_cells(b, ko, bid, W), arena, slots);
        if (cls >= 0) atomicAdd(&wk.count[cls], 1);
    }
}
__global__ void k_flood_scatter_ranked(BlobInfo b, int W, FloodWork wk, int arena, int slots) {
    int n = blockIdx.y;
    long long ko = (long long)n * b.KS;
    int B = b.count[n];
    for (int bid = 1 + blockIdx.x * blockDim.x + threadIdx.x; bid <= B; bid += gridDim.x * blockDim.x) {
        long long item = ((long long)n << 32) | (unsigned)bid;
        if (blob_is_huge(b, ko, bid, W)) { wk.ovf[atomicAdd(wk.ngen + 1, 1)] = item; continue; }
        int cls = blob_class(blob_cells(b, ko, bid, W), arena, slots);
        if (cls >= 0) wk.items[wk.offset[cls] + atomicAdd(&wk.fill[cls], 1)] = item;
        else wk.gen[atomicAdd(wk.ngen, 1)] = item;
    }
}

// one blob per CTA at a time, ranked levels, all arrays sized by the blob (levels < cells)
__device__ __forceinline__ void general_drain_ranked(const Geom& g, const unsigned short* __restrict__ level,
                                                     const int* __restrict__ par, const BlobInfo& b, const long long* list,
                                                     int count, int* cursor, int32_t* out) {
    __shared__ int s_item;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    unsigned short* lab = reinterpret_cast<unsigned short*>(ws_smem);
    unsigned short* nxs = lab + WR_GEN_CAP;
    unsigned short* lvl = nxs;                       // level and FIFO link share a field (see stage_copy)
    unsigned short* head = nxs + WR_GEN_CAP;
    unsigned short* tail = head + WR_GEN_CAP;
    const int W = g.W;
    for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) s_item = atomicAdd(cursor, 1);
        __syncthreads();
        const int k = s_item;
        if (k >= count) break;
        const long long item = list[k];
        const int n = (int)(item >> 32), bid = (int)(item & 0xffffffffll);
        const long long base = (long long)n * g.P, ko = (long long)n * b.KS;
        const int root = b.root[ko + bid];
        const int y0 = root / W, x0 = b.xmin[ko + bid];
        const int w = b.xmax[ko + bid] - x0 + 1, h = b.ymax[ko + bid] - y0 + 1;
        const int cells = (w + 2) * (h + 2);
        for (int i = threadIdx.x; i < cells; i += blockDim.x) { head[i] = (unsigned short)WS_END; tail[i] = (unsigned short)WS_END; }
        stage_copy(threadIdx.x, blockDim.x, W, level + base, InForest{par + base, root}, out + base, root, y0, x0, w, h, lab, lvl);
        __syncthreads();
        if (warp == 0) {
            int vmin, vmax, vsmin;
            link_seeds(lane, cells, lab, nxs, lvl, head, tail, BucketDirect{0}, vmin, vmax, vsmin);
            __syncwarp();
            if (lane == 0 && vsmin <= vmax) lane_flood(w + 2, vsmin, vmax, lab, nxs, lvl, head, tail, BucketDirect{0});
        }
        __syncthreads();
        stage_writeback(threadIdx.x, blockDim.x, W, out + base, y0, x0, w, h, lab);
    }
}

template <int WARPS, int ARENA, int SLOTS>
__global__ void __launch_bounds__(32 * WARPS, 1)
k_ws_flood_ranked(Geom g, const unsigned short* __restrict__ level, const int* __restrict__ par, BlobInfo b, FloodWork wk,
                  int32_t* out, int gen_first) {
    const int ngen = wk.ngen[0];
    if ((int)blockIdx.x < min(gen_first, ngen)) general_drain_ranked(g, level, par, b, wk.gen, ngen, wk.gcursor, out);
    __syncthreads();
    {
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
        unsigned short* lab = reinterpret_cast<unsigned short*>(ws_smem) + (size_t)warp * ARENA * 4;
        unsigned short* nxs = lab + ARENA;
        unsigned short* lvl = nxs;
        unsigned short* head = nxs + ARENA;
        unsigned short* tail = head + ARENA;
        const int W = g.W;
        for (int cls = 0; cls < SLOTS; ++cls) {
            const int cap = ARENA / (cls + 1), slots = cls + 1;
            const int cnt = wk.count[cls];
            const long long* list = wk.items + wk.offset[cls];
            for (;;) {
                int k0 = 0;
                if (lane == 0) k0 = atomicAdd(&wk.cursor[cls], slots);
                k0 = __shfl_sync(FULL, k0, 0);
                if (k0 >= cnt) break;
                const int m = min(slots, cnt - k0);
                int mn = 0, mroot = 0, my0 = 0, mx0 = 0, mw = 0, mh = 0;
                if (lane < m) {
                    const long long item = list[k0 + lane];
                    mn = (int)(item >> 32);
                    const int bid = (int)(item & 0xffffffffll);
                    const long long ko = (long long)mn * b.KS;
                    mroot = b.root[ko + bid];
                    my0 = mroot / W; mx0 = b.xmin[ko + bid];
                    mw = b.xmax[ko + bid] - mx0 + 1; mh = b.ymax[ko + bid] - my0 + 1;
                }
                for (int i = lane; i < m * cap; i += 32) { head[i] = (unsigned short)WS_END; tail[i] = (unsigned short)WS_END; }
                unsigned single = 0;
                for (int s = 0; s < m; ++s) {
                    const int n = __shfl_sync(FULL, mn, s), root = __shfl_sync(FULL, mroot, s);
                    const int y0 = __shfl_sync(FULL, my0, s), x0 = __shfl_sync(FULL, mx0, s);
                    const int w = __shfl_sync(FULL, mw, s), h = __shfl_sync(FULL, mh, s);
                    const long long base = (long long)n * g.P;
                    const SeedStats st = stage_copy(lane, 32, W, level + base, InForest{par + base, root}, out + base, root, y0, x0, w, h,
                                                    lab + s * cap, lvl + s * cap);
                    __syncwarp();
                    if (fill_if_single_marker(lane, st, (w + 2) * (h + 2), lab + s * cap)) single |= 1u << s;
                }
                __syncwarp();
                int lmax = -1, smin = WS_LVL_NONE;              // of slot `lane`
                for (int s = 0; s < m; ++s) {
                    if ((single >> s) & 1u) continue;
                    const int w = __shfl_sync(FULL, mw, s), h = __shfl_sync(FULL, mh, s);
                    int vmin, vmax, vsmin;
                    link_seeds(lane, (w + 2) * (h + 2), lab + s * cap, nxs + s * cap, lvl + s * cap, head, tail,
                               BucketDirect{s * cap}, vmin, vmax, vsmin);
                    if (lane == s) { lmax = vmax; smin = vsmin; }
                }
                __syncwarp();
                if (lane < m && smin <= lmax)
                    lane_flood(mw + 2, smin, lmax, lab + lane * cap, nxs + lane * cap, lvl + lane * cap, head, tail,
                               BucketDirect{lane * cap});
                __syncwarp();
                for (int s = 0; s < m; ++s) {
                    const int n = __shfl_sync(FULL, mn, s);
                    const int y0 = __shfl_sync(FULL, my0, s), x0 = __shfl_sync(FULL, mx0, s);
                    const int w = __shfl_sync(FULL, mw, s), h = __shfl_sync(FULL, mh, s);
                    stage_writeback(lane, 32, W, out + (long long)n * g.P, y0, x0, w, h, lab + s * cap);
                }
                __syncwarp();
            }
        }
    }
    if (ngen > 0) general_drain_ranked(g, level, par, b, wk.gen, ngen, wk.gcursor, out);
}

// ---- fp64 values: binary heap keyed (value, age, index) -------------------------------------------------
struct __align__(16) HeapItem { double v; unsigned age; int idx; };

__device__ __forceinline__ bool heap_less(const HeapItem& a, const HeapItem& b) {
    if (a.v != b.v) return a.v < b.v;
    if (a.age != b.age) return a.age < b.age;
    return a.idx < b.idx;
}
__device__ __forceinline__ void heap_push(HeapItem* h, int& sz, HeapItem it) {
    int i = sz++;
    while (i > 0) {
        int p = (i - 1) >> 1;
        HeapItem hp = h[p];
        if (!heap_less(it, hp)) break;
        h[i] = hp;
        i = p;
    }
    h[i] = it;
}
__device__ __forceinline__ HeapItem heap_pop(HeapItem* h, int& sz) {
    HeapItem top = h[0];
    HeapItem last = h[--sz];
    int i = 0;
    for (;;) {
        int l = 2 * i + 1;
        if (l >= sz) break;
        HeapItem c = h[l];
        if (l + 1 < sz) {
            HeapItem r = h[l + 1];
            if (heap_less(r, c)) { c = r; l = l + 1; }
        }
        if (!heap_less(c, last)) break;
        h[i] = c;
        i = l;
    }
    if (sz > 0) h[i] = last;
    return top;
}

// one warp per listed blob, list[0 .. *nlist) (persistent grid; `cursor` hands out the items)
__global__ void __launch_bounds__(TISEG_THREADS)
k_ws_flood_f64(Geom g, const double* __restrict__ image, const int* __restrict__ par, BlobInfo b, int* cursor,
               const long long* __restrict__ list, const int* __restrict__ nlist, HeapItem* heap, int32_t* out) {
    const int lane = threadIdx.x & 31;
    const int W = g.W, H = g.H;
    for (;;) {
        int k = 0;
        if (lane == 0) k = atomicAdd(cursor, 1);
        k = __shfl_sync(FULL, k, 0);
        if (k >= *nlist) break;
        const int n = (int)(list[k] >> 32), bid = (int)(list[k] & 0xffffffffll);
        const long long base = (long long)n * g.P, ko = (long long)n * b.KS;
        const double* I = image + base;
        const int* tp = par + base;
        int32_t* o = out + base;
        const int root = b.root[ko + bid];
        const int y0 = root / W, y1 = b.ymax[ko + bid], x0 = b.xmin[ko + bid], x1 = b.xmax[ko + bid];
        HeapItem* h = heap + base + b.off[ko + bid];
        int sz = 0;
        for (int y = y0; y <= y1; ++y) {
            for (int xb = x0; xb <= x1; xb += 32) {
                int x = xb + lane;
                bool seed = false;
                double v = 0.0;
                if (x <= x1) {
                    int idx = y * W + x;
                    if (tp[idx] == root && o[idx] != 0) { seed = true; v = I[idx]; }
                }
                unsigned m = __ballot_sync(FULL, seed);
                while (m) {
                    int src = __ffs(m) - 1;
                    m &= m - 1;
                    double sv = __shfl_sync(FULL, v, src);
                    if (lane == 0) { HeapItem it; it.v = sv; it.age = 0u; it.idx = y * W + xb + src; heap_push(h, sz, it); }
                }
            }
        }
        if (lane == 0) {
            unsigned age = 0;
            while (sz > 0) {
                HeapItem e = heap_pop(h, sz);
                const int pix = e.idx;
                const int lab = o[pix];
                const int y = pix / W, x = pix - y * W;
                const int nb[4] = {pix - W, pix - 1, pix + 1, pix + W};
                const bool ok[4] = {y > 0, x > 0, x + 1 < W, y + 1 < H};
                int pv[4], ov[4];
                double vv[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    pv[k] = -1; ov[k] = 1; vv[k] = 0.0;
                    if (ok[k]) { pv[k] = tp[nb[k]]; ov[k] = o[nb[k]]; vv[k] = I[nb[k]]; }
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if (pv[k] >= 0 && ov[k] == 0) {
                        o[nb[k]] = lab;
                        HeapItem it; it.v = vv[k]; it.age = ++age; it.idx = nb[k];
                        heap_push(h, sz, it);
                    }
                }
            }
        }
        __syncwarp();
    }
}

int ws_seed(tiseg_ctx* c, const Geom& g, const int32_t* markers, const int* par, int32_t* out) {
    long long total = (long long)g.N * g.P;
    TISEG_LAUNCH(c, k_ws_seed, flat4_grid(total), TISEG_THREADS, 0, total, markers, par, out, aligned16(markers, par, out));
    return TISEG_OK;
}

int blobs_describe(tiseg_ctx* c, const Geom& g, const int* par, const int* rank, const unsigned* root_bits, BlobInfo& b,
                   bool want_offsets) {
    TISEG_LAUNCH(c, k_blob_init, dim3(8, g.N), 256, 0, b, g.W);
    TISEG_LAUNCH(c, k_blob_roots, dim3((unsigned)(((long long)g.H * g.SEG + TISEG_THREADS - 1) / TISEG_THREADS), g.N), TISEG_THREADS, 0,
                 g, root_bits, rank, b);
    TISEG_LAUNCH(c, k_blob_bbox, quad_grid(g), TISEG_THREADS, 0, g, par, rank, b, (g.W % 4 == 0) && aligned16(par));
    if (want_offsets) TISEG_LAUNCH(c, k_blob_offsets, g.N, 256, 0, b);
    return TISEG_OK;
}

template <bool MASKED>
static int watershed_u8_any(tiseg_ctx* c, const Geom& g, const uint8_t* image, const BlobMember& bm, const BlobInfo& b, int32_t* out) {
    const int N = g.N;
    const size_t max_blobs = (size_t)N * ((size_t)g.P / 2 + 1);      // a checkerboard is the worst case
    FloodWork wk;
    wk.items = ws<long long>(c, max_blobs);
    wk.gen = ws<long long>(c, max_blobs);
    wk.ovf = nullptr;
    int* ints = ws<int>(c, WK_INTS + 2 * (size_t)N + 1);
    int* next = ws<int>(c, (size_t)N * g.P);
    int* gheads = ws<int>(c, (size_t)c->sm_count * 512);
    if (!wk.items || !wk.gen || !ints || !next || !gheads) return TISEG_ERR_CUDA;
    wk.count = ints; wk.offset = ints + WS_MAXCLS; wk.fill = ints + 2 * WS_MAXCLS; wk.cursor = ints + 3 * WS_MAXCLS;
    wk.ngen = ints + 4 * WS_MAXCLS; wk.gcursor = wk.ngen + 2;
    int* huge = ints + WK_INTS;                 // tiles with a blob that is flooded in global memory
    TISEG_TRY(zero(c, ints, (WK_INTS + 2 * (size_t)N + 1) * sizeof(int)));
    static_assert(WP_SMEM_BYTES + 64 <= 232448, "shared memory");
    TISEG_LAUNCH(c, k_flood_count, dim3(8, g.N), 256, 0, b, g.W, wk, WP_ARENA, WS_MAXCLS);
    TISEG_LAUNCH(c, k_flood_offsets, 1, 32, 0, wk);
    TISEG_LAUNCH(c, k_flood_scatter, dim3(8, g.N), 256, 0, b, g.W, wk, WP_ARENA, WS_MAXCLS, (long long)WP_GEN_CAP, MASKED ? huge : (int*)nullptr);
    // mask mode: the label map holds the seeds and is otherwise unwritten; the flood in global memory reads it
    if (MASKED) {
        Geom gh = listed_geom(g, huge + N, huge + 2 * N);
        const BitPlanes mp = {const_cast<unsigned*>(bm.mask_bits), nullptr, nullptr, nullptr, nullptr};
        TISEG_LAUNCH(c, k_huge_clean, dim3((unsigned)(((long long)g.H * g.SEG + TISEG_THREADS - 1) / TISEG_THREADS), 1), TISEG_THREADS, 0,
                     gh, mp, bm.bpar, bm.brank, b, bm.seed_bits, (long long)WP_GEN_CAP, out);
    }
    if (!c->smem_flood_u8[MASKED]) {
        TISEG_CHECK(cudaFuncSetAttribute(k_ws_flood_par<MASKED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)WP_SMEM_BYTES));
        c->smem_flood_u8[MASKED] = true;
    }
    TISEG_LAUNCH_AS(c, "k_ws_flood_par", (k_ws_flood_par<MASKED>), c->sm_count, 32 * WP_WARPS, WP_SMEM_BYTES, g, image, bm, b,
                    wk, next, gheads, out);
    return TISEG_OK;
}

int watershed_u8_dev(tiseg_ctx* c, const Geom& g, const uint8_t* image, const int* par, const int* rank,
                     const BlobInfo& b, int32_t* out) {
    (void)rank;
    BlobMember bm;
    bm.par = par; bm.mask_img = nullptr; bm.seed_blob = nullptr; bm.seed_bits = nullptr; bm.mask_bits = nullptr; bm.bpar = nullptr; bm.brank = nullptr;
    return watershed_u8_any<false>(c, g, image, bm, b, out);
}

int watershed_u8_masked_dev(tiseg_ctx* c, const Geom& g, const uint8_t* image, const BlobMember& bm, const BlobInfo& b, int32_t* out) {
    return watershed_u8_any<true>(c, g, image, bm, b, out);
}

int blobs_ccl(tiseg_ctx* c, const Geom& g, const BitPlanes& planes, int* par, int* rank, int* first, BlobInfo& b) {
    const int N = g.N, KS = g.P + 1;
    const size_t ks = (size_t)N * KS, words = (size_t)N * g.H * g.SEG;
    int* count = ws<int>(c, (size_t)N);
    b.root = ws<int>(c, ks); b.ymax = ws<int>(c, ks); b.xmin = ws<int>(c, ks); b.xmax = ws<int>(c, ks);
    b.area = ws<int>(c, ks); b.off = nullptr; b.lmin = ws<int>(c, ks); b.lmax = ws<int>(c, ks);
    b.KS = KS; b.count = count; b.first = first;
    unsigned* lbits = ws<unsigned>(c, words);
    unsigned* fbits = ws<unsigned>(c, words);
    if (!count || !b.root || !b.ymax || !b.xmin || !b.xmax || !b.area || !b.lmin || !b.lmax || !lbits || !fbits) return TISEG_ERR_CUDA;
    TISEG_TRY(bitccl_build(c, g, planes, 1, par, lbits, fbits));           // 4-connected components of the mask
    TISEG_TRY(rank_from_bits(c, g, fbits, rank, count));
    const dim3 wg((unsigned)(((long long)g.H * g.SEG + TISEG_THREADS - 1) / TISEG_THREADS), (unsigned)N);
    TISEG_LAUNCH(c, k_blob_init, dim3(8, N), 256, 0, b, g.W);
    TISEG_LAUNCH(c, k_blob_roots, wg, TISEG_THREADS, 0, g, fbits, rank, b);
    return TISEG_OK;
}

int blobs_boxes_fill(tiseg_ctx* c, const Geom& g, const BitPlanes& planes, const int* par, const int* rank, const BlobInfo& b,
                     int32_t* out) {
    const dim3 wg((unsigned)(((long long)g.H * g.SEG + TISEG_THREADS - 1) / TISEG_THREADS), (unsigned)g.N);
    TISEG_LAUNCH(c, k_blob_runs, wg, TISEG_THREADS, 0, g, planes, par, rank, b, out);
    return TISEG_OK;
}

int watershed_f64_dev(tiseg_ctx* c, const Geom& g, const double* image, const int* par, const int* rank,
                      const BlobInfo& b, int32_t* out) {
    (void)rank;
    const int N = g.N;
    HeapItem* heap = ws<HeapItem>(c, (size_t)N * g.P);
    if (!heap || !b.off) return TISEG_ERR_CUDA;
    // ranked levels per blob, then the bucket flood in shared memory
    constexpr int WARPS = 7, ARENA = 3840, SLOTS = 16;
    constexpr size_t MULTI = (size_t)WARPS * ARENA * 8, GEN = (size_t)WR_GEN_CAP * 8;
    constexpr size_t SMEM = MULTI > GEN ? MULTI : GEN;
    static_assert(SMEM + 64 <= 232448, "shared memory");
    const size_t max_blobs = (size_t)N * ((size_t)g.P / 2 + 1);
    unsigned short* level = ws<unsigned short>(c, (size_t)N * g.P);
    int* prefix = ws<int>(c, (size_t)N + 1);
    FloodWork wk;
    wk.items = ws<long long>(c, max_blobs);
    wk.gen = ws<long long>(c, max_blobs);
    wk.ovf = ws<long long>(c, max_blobs);
    int* ints = ws<int>(c, WK_INTS);
    if (!level || !prefix || !wk.items || !wk.gen || !wk.ovf || !ints) return TISEG_ERR_CUDA;
    wk.count = ints; wk.offset = ints + WS_MAXCLS; wk.fill = ints + 2 * WS_MAXCLS; wk.cursor = ints + 3 * WS_MAXCLS;
    wk.ngen = ints + 4 * WS_MAXCLS; wk.gcursor = wk.ngen + 2;
    TISEG_TRY(zero(c, ints, WK_INTS * sizeof(int)));
    constexpr size_t RK_SMALL = (size_t)WR_SORT_SMALL * 10, RK_LARGE = (size_t)WR_SORT_MAX * 10;
    if (!c->smem_flood_f64) {
        TISEG_CHECK(cudaFuncSetAttribute(k_rank_blobs<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RK_LARGE));
        TISEG_CHECK(cudaFuncSetAttribute((k_ws_flood_ranked<WARPS, ARENA, SLOTS>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
        c->smem_flood_f64 = true;
    }
    TISEG_LAUNCH(c, k_blob_prefix, 1, 32, 0, b.count, N, prefix);
    TISEG_LAUNCH(c, k_rank_blobs<false>, c->sm_count * 16, 128, RK_SMALL, g, image, par, b, prefix, level);
    TISEG_LAUNCH(c, k_rank_blobs<true>, c->sm_count, 1024, RK_LARGE, g, image, par, b, prefix, level);
    TISEG_LAUNCH(c, k_flood_count_ranked, dim3(8, N), 256, 0, b, g.W, wk, ARENA, SLOTS);
    TISEG_LAUNCH(c, k_flood_offsets, 1, 32, 0, wk);
    TISEG_LAUNCH(c, k_flood_scatter_ranked, dim3(8, N), 256, 0, b, g.W, wk, ARENA, SLOTS);
    const int gen_first = c->sm_count >= 8 ? c->sm_count / 4 : 1;
    TISEG_LAUNCH(c, (k_ws_flood_ranked<WARPS, ARENA, SLOTS>), c->sm_count, 32 * WARPS, SMEM, g, level, par, b, wk, out, gen_first);
    // blobs too large to rank / stage: the heap flood in global memory (persistent grid; exits at once if there are none)
    TISEG_LAUNCH(c, k_ws_flood_f64, dim3(c->sm_count, 1), TISEG_THREADS, 0, g, image, par, b, wk.gcursor + 1,
                 (const long long*)wk.ovf, (const int*)(wk.ngen + 1), heap, out);
    return TISEG_OK;
}

template <class T>
static int watershed_entry(tiseg_ctx* c, const T* image, const int32_t* markers, const uint8_t* mask, int N, int H,
                           int W, int32_t* out) {
    if (!c || !image || !markers || !out) { set_error("tiseg_watershed: bad argument"); return TISEG_ERR_ARG; }
    Call call(c, sizeof(T) == 8 ? "tiseg_watershed_f64" : "tiseg_watershed_u8", N, H, W);
    const Geom& g = call.g;
    const T* d_img = call.in(image, call.total);
    const int32_t* d_mk = call.in(markers, call.total);
    const uint8_t* d_mask = call.in(mask, call.total);
    int32_t* d_out = call.out(out, call.total);
    TISEG_TRY(call.status());
    int* par = ws<int>(c, call.total);
    int* rank = ws<int>(c, call.total);
    if (!par || !rank) return TISEG_ERR_CUDA;
    BlobInfo b;
    constexpr bool F64 = sizeof(T) == 8;
    if (d_mask) TISEG_TRY(blobs_build(c, g, ImgMaskU8{d_mask}, par, rank, b, F64));
    else        TISEG_TRY(blobs_build(c, g, ImgAll{}, par, rank, b, F64));
    TISEG_TRY(ws_seed(c, g, d_mk, par, d_out));
    if constexpr (F64) TISEG_TRY(watershed_f64_dev(c, g, (const double*)d_img, par, rank, b, d_out));
    else               TISEG_TRY(watershed_u8_dev(c, g, (const uint8_t*)d_img, par, rank, b, d_out));
    return call.finish();
}

}  // namespace tiseg

using namespace tiseg;

extern "C" {

int tiseg_watershed_u8(tiseg_ctx* c, const uint8_t* image, const int32_t* markers, const uint8_t* mask, int N, int H,
                       int W, int32_t* out) {
    return watershed_entry<uint8_t>(c, image, markers, mask, N, H, W, out);
}

int tiseg_watershed_f64(tiseg_ctx* c, const double* image, const int32_t* markers, const uint8_t* mask, int N, int H,
                        int W, int32_t* out) {
    return watershed_entry<double>(c, image, markers, mask, N, H, W, out);
}

}  // extern "C"
