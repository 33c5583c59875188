// K12 / K13 — evaluation kernels: GT x pred pair-overlap histogram -> AJI and PQ, semantic counts.
//
//   tiseg_pair_metrics_bin  replaces pre_eval_bin_aji + pre_eval_bin_pq (tiseg/utils/inst_metrics.py:10-92,
//                           138-229) including the measure.label relabelling they start with.
//   tiseg_sem_counts        replaces pre_eval_all_semantic_metric (tiseg/utils/sem_metrics.py:16-53).
//
// The reference materialises one full-image mask per instance (O(K*P)); here the non-zero entries of the
// [Ng, Np] intersection matrix are accumulated in one pass into a per-tile open-addressing hash table keyed
// by (gt id, pred id) — one atomic per horizontal RUN of equal pairs (warp ballot), not per pixel — and
// everything downstream works on the O(K) non-zero pairs.  Counts are exact integers; the only floating
// point is the fp64 IoU used for argmax / thresholding, evaluated with the reference's expressions.
#include "bitccl.cuh"
#include "ccl.cuh"

namespace tiseg {

// Two tables: a small one (instances are compact: O(K) pairs) that every batch tries first, and an
// always-sufficient one (2P slots per tile: a pair needs a pixel) that is zeroed and filled ON THE DEVICE only if the
// small one overflowed — no host round trip decides.  `view()` gives the table in force.
struct PairTabView {
    unsigned long long* key;   // [N, cap]  (g << 32 | p), 0 = empty
    int* cnt;                  // [N, cap]
    int cap;                   // power of two
};
struct PairTab {
    PairTabView small, big;
    int* overflow;             // [1] set by the first accumulation pass
    __device__ __forceinline__ PairTabView view() const { return *overflow ? big : small; }
};

__device__ __forceinline__ unsigned pair_hash(unsigned g, unsigned p) {
    unsigned h = g * 0x9E3779B1u ^ p * 0x85EBCA6Bu;
    h ^= h >> 15; h *= 0x2C1B3C6Du; h ^= h >> 12;
    return h;
}

__device__ __forceinline__ void pair_add(const PairTabView& t, int n, unsigned g, unsigned p, int len, int* overflow) {
    unsigned long long k = ((unsigned long long)g << 32) | p;
    unsigned long long* keys = t.key + (long long)n * t.cap;
    unsigned s = pair_hash(g, p) & (t.cap - 1);
    for (int probe = 0; probe < t.cap; ++probe) {
        unsigned long long cur = keys[s];
        if (cur == 0) {
            cur = atomicCAS(&keys[s], 0ull, k);
            if (cur == 0) cur = k;                         // we claimed the slot
        }
        if (cur == k) { atomicAdd(&t.cnt[(long long)n * t.cap + s], len); return; }
        s = (s + 1) & (t.cap - 1);
    }
    *overflow = 1;
}

__device__ __forceinline__ int pair_lookup(const PairTabView& t, int n, unsigned g, unsigned p) {
    unsigned long long k = ((unsigned long long)g << 32) | p;
    const unsigned long long* keys = t.key + (long long)n * t.cap;
    unsigned s = pair_hash(g, p) & (t.cap - 1);
    for (int probe = 0; probe < t.cap; ++probe) {
        unsigned long long cur = keys[s];
        if (cur == k) return t.cnt[(long long)n * t.cap + s];
        if (cur == 0) return 0;
        s = (s + 1) & (t.cap - 1);
    }
    return 0;
}

// per-instance state, dense by id with a per-tile stride of KS = P + 1 entries (only the first K+1 are touched)
struct InstState {
    int* area_g; int* area_p;          // [N, KS]
    unsigned long long* best;          // [N, KS] fp64 bits of the best AJI IoU per gt id
    int* bestp;                        // [N, KS] lowest pred id reaching `best`
    uint8_t* used;                     // [N, KS] pred id chosen by some gt
    double* pqiou;                     // [N, KS] IoU of the (unique) PQ match of a gt id, 0 = none
    const int* ng; const int* np;      // [N] number of components (ids 1..K)
    int KS;
    // class of every component (NULL = binary evaluation: every component is class 1), C class slots
    const uint8_t* cls_g; const uint8_t* cls_p;
    int C;
    __device__ __forceinline__ int class_g(long long o, unsigned id) const { return cls_g ? cls_g[o + id] : 1; }
    __device__ __forceinline__ int class_p(long long o, unsigned id) const { return cls_p ? cls_p[o + id] : 1; }
};

__global__ void k_inst_init(InstState s, int areas) {
    int n = blockIdx.y;
    long long o = (long long)n * s.KS;
    int ng = s.ng[n], np = s.np[n];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i <= ng; i += gridDim.x * blockDim.x) {
        if (areas) s.area_g[o + i] = 0;
        s.best[o + i] = 0ull; s.bestp[o + i] = 0x7fffffff; s.pqiou[o + i] = 0.0;
    }
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i <= np; i += gridDim.x * blockDim.x) {
        if (areas) s.area_p[o + i] = 0;
        s.used[o + i] = 0;
    }
}

// clears the always-sufficient table for the redo (persistent grid; exits at once unless the small table overflowed)
__global__ void __launch_bounds__(TISEG_THREADS) k_pair_zero_big(PairTab t, PairTab u, int N) {
    if (!*t.overflow) return;
    const long long total = (long long)N * t.big.cap;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        t.big.key[i] = 0ull; t.big.cnt[i] = 0;
        if (u.big.key != t.big.key) { u.big.key[i] = 0ull; u.big.cnt[i] = 0; }
    }
}

// =====================================================================================================================
// Pair table from bit planes (tiseg_pair_metrics_*; bitccl.cuh).
//
// measure.label of both maps (inst_metrics.py:12-13) only serves to IDENTIFY the components the pair matrix is indexed
// by; no per-pixel label map is needed.  Both instance maps are read ONCE (k_eqbits, 4 B/px each) into equality bit
// planes; the union-find, the cross-tile merges, the final-root bitmaps and their raster-order ranks work on words and
// runs; and the pair histogram is accumulated by one thread per 32-pixel word from the planes of the two maps: a piece
// of a row on which both labels are constant is delimited with bit operations, the component ids of its two runs are
// looked up at the run starts, and one set of atomics is posted per piece (areas by id + the (gt, pred) hash table).
// =====================================================================================================================

// p: planes of 2N tile-batch entries (gt tiles, then pred tiles); par / rank: [2N, P]
template <bool BIG>
__global__ void __launch_bounds__(TISEG_THREADS)
k_pair_bits(Geom g, BitPlanes p, const int* __restrict__ par, const int* __restrict__ rank, InstState s, PairTab t, int* lost) {
    if (BIG && !*t.overflow) return;
    const long long words = (long long)g.H * g.SEG;
    const long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= words) return;
    const int n = blockIdx.y, N = gridDim.y;
    const long long wg = (long long)n * words, wp = (long long)(N + n) * words;
    const unsigned Fg = p.F[wg + w], Fp = p.F[wp + w];
    const unsigned fany = Fg | Fp;
    if (!fany) return;
    const int y = (int)(w / g.SEG), seg = (int)(w - (long long)y * g.SEG);
    const unsigned Cg = p.C[wg + w], Cp = p.C[wp + w];
    const unsigned cg = seg > 0 ? p.F[wg + w - 1] >> 31 : 0u, cp = seg > 0 ? p.F[wp + w - 1] >> 31 : 0u;
    // "same label as the pixel to the left" on each side (background next to background counts as the same label)
    const unsigned same_g = Cg | (~Fg & ~((Fg << 1) | cg)), same_p = Cp | (~Fp & ~((Fp << 1) | cp));
    const unsigned starts = fany & (~(same_g & same_p) | 1u);            // pieces are also cut at the word boundary
    const PairTabView tv = BIG ? t.big : t.small;
    int* ovf = BIG ? lost : t.overflow;
    const long long o = (long long)n * s.KS;
    const long long pg = (long long)n * g.P, pp = (long long)(N + n) * g.P;
    for (unsigned m = starts; m; m &= m - 1) {
        const int b = __ffs(m) - 1;
        const unsigned rest = b == 31 ? 0u : (starts | ~fany) >> (b + 1);
        const int len = rest ? __ffs(rest) : 32 - b;
        const int x = seg * 32 + b;
        int gid = 0, pid = 0;
        if ((Fg >> b) & 1u) gid = rank[pg + find_ro(par + pg, bit_node_of(p, g, wg, y, x))];
        if ((Fp >> b) & 1u) pid = rank[pp + find_ro(par + pp, bit_node_of(p, g, wp, y, x))];
        if (!BIG) {
            if (gid) atomicAdd(&s.area_g[o + gid], len);
            if (pid) atomicAdd(&s.area_p[o + pid], len);
        }
        if (gid && pid) pair_add(tv, n, (unsigned)gid, (unsigned)pid, len, ovf);
    }
}

// pass A over the table: best AJI IoU per gt (atomicMax on fp64 bits: positive doubles order like integers),
// and the PQ matches (IoU > 0.5 is unique per gt and per pred)
__global__ void k_pair_best(PairTab tt, InstState s, int* tp, double match_iou) {
    const PairTabView t = tt.view();
    int n = blockIdx.y;
    for (int slot = blockIdx.x * blockDim.x + threadIdx.x; slot < t.cap; slot += gridDim.x * blockDim.x) {
    unsigned long long k = t.key[(long long)n * t.cap + slot];
    if (!k) continue;
    unsigned gid = (unsigned)(k >> 32), pid = (unsigned)k;
    long long o = (long long)n * s.KS;
    int cg = s.class_g(o, gid);
    if (cg == 0 || cg != s.class_p(o, pid)) continue;       // only pairs inside one class meet (inst_metrics.py:112-122)
    double inter = (double)t.cnt[(long long)n * t.cap + slot];
    double tot = (double)s.area_g[o + gid] + (double)s.area_p[o + pid];
    double iou_aji = inter / ((tot - inter) + 1.0e-6);      // inst_metrics.py:69
    atomicMax(&s.best[o + gid], (unsigned long long)__double_as_longlong(iou_aji));
    double iou_pq = inter / (tot - inter);                  // inst_metrics.py:194
    if (iou_pq > match_iou) { s.pqiou[o + gid] = iou_pq; atomicAdd(&tp[n * s.C + cg], 1); }     // inst_metrics.py:197-203, match_iou >= 0.5
    }
}

// pass B: np.argmax tie rule — the lowest pred id among those reaching the best IoU (inst_metrics.py:74)
__global__ void k_pair_argbest(PairTab tt, InstState s) {
    const PairTabView t = tt.view();
    int n = blockIdx.y;
    for (int slot = blockIdx.x * blockDim.x + threadIdx.x; slot < t.cap; slot += gridDim.x * blockDim.x) {
    unsigned long long k = t.key[(long long)n * t.cap + slot];
    if (!k) continue;
    unsigned gid = (unsigned)(k >> 32), pid = (unsigned)k;
    long long o = (long long)n * s.KS;
    int cg = s.class_g(o, gid);
    if (cg == 0 || cg != s.class_p(o, pid)) continue;
    double inter = (double)t.cnt[(long long)n * t.cap + slot];
    double tot = (double)s.area_g[o + gid] + (double)s.area_p[o + pid];
    double iou_aji = inter / ((tot - inter) + 1.0e-6);
    if ((unsigned long long)__double_as_longlong(iou_aji) == s.best[o + gid]) atomicMin(&s.bestp[o + gid], (int)pid);
    }
}

// add (I, U) of one instance to its class slot; warps whose lanes all share one class (always, in the binary
// evaluation) combine by shuffle first so the slot sees one atomic per warp
__device__ __forceinline__ void add_iu(unsigned long long* IU, int n, int C, int cls, unsigned long long I,
                                       unsigned long long U, bool active) {
    int key = active ? cls : -1;
    int kmax = key;
    for (int d = 16; d; d >>= 1) kmax = max(kmax, __shfl_xor_sync(0xffffffffu, kmax, d));
    bool uniform = __all_sync(0xffffffffu, key == kmax || key == -1);
    if (uniform) {
        if (kmax < 0) return;
        for (int d = 16; d; d >>= 1) { I += __shfl_down_sync(0xffffffffu, I, d); U += __shfl_down_sync(0xffffffffu, U, d); }
        if ((threadIdx.x & 31) == 0) {
            if (I) atomicAdd(&IU[((long long)n * C + kmax) * 2], I);
            if (U) atomicAdd(&IU[((long long)n * C + kmax) * 2 + 1], U);
        }
    } else if (active) {
        if (I) atomicAdd(&IU[((long long)n * C + cls) * 2], I);
        if (U) atomicAdd(&IU[((long long)n * C + cls) * 2 + 1], U);
    }
}

// pass C: per gt — paired inter / union, or its own area when nothing overlaps (inst_metrics.py:76-87);
// class-0 instances only contribute their area to union[0] (inst_metrics.py:105-110)
__global__ void k_aji_gt(PairTab tt, InstState s, unsigned long long* IU) {
    const PairTabView t = tt.view();
    int n = blockIdx.y;
    long long o = (long long)n * s.KS;
    int ng = s.ng[n];
    int span = gridDim.x * blockDim.x;
    for (int g0 = 1 + blockIdx.x * blockDim.x; g0 <= ng; g0 += span) {     // warp-uniform trip count
        int gid = g0 + threadIdx.x;
        bool act = gid <= ng;
        unsigned long long I = 0, U = 0;
        int cls = 0;
        if (act) {
            cls = s.class_g(o, gid);
            int ag = s.area_g[o + gid];
            if (cls != 0 && s.best[o + gid] != 0ull) {
                int pid = s.bestp[o + gid];
                int inter = pair_lookup(t, n, gid, pid);
                I = inter;
                U = (unsigned long long)(ag + s.area_p[o + pid] - inter);
                s.used[o + pid] = 1;
            } else {
                U = ag;
            }
        }
        add_iu(IU, n, s.C, cls, I, U, act);
    }
}

// pass D: preds never chosen by any gt add their area to the union (inst_metrics.py:88-90)
__global__ void k_aji_pred(InstState s, unsigned long long* IU) {
    int n = blockIdx.y;
    long long o = (long long)n * s.KS;
    int np = s.np[n];
    int span = gridDim.x * blockDim.x;
    for (int p0 = 1 + blockIdx.x * blockDim.x; p0 <= np; p0 += span) {
        int pid = p0 + threadIdx.x;
        bool act = pid <= np;
        unsigned long long U = 0;
        int cls = 0;
        if (act) {
            cls = s.class_p(o, pid);
            if (cls == 0 || !s.used[o + pid]) U = s.area_p[o + pid];
        }
        add_iu(IU, n, s.C, cls, 0ull, U, act);
    }
}

// numpy's pairwise summation (numpy/core/src/umath/loops_utils.h.src, DOUBLE_pairwise_sum): what
// `paired_iou.sum()` (inst_metrics.py:227) evaluates, reproduced so iou_sum is bit-identical.
__device__ __forceinline__ double np_pairwise_leaf(const double* a, int n) {   // n <= 128
    if (n < 8) {
        double r = 0.0;
        for (int i = 0; i < n; ++i) r += a[i];
        return r;
    }
    double r[8];
    for (int j = 0; j < 8; ++j) r[j] = a[j];
    int i;
    for (i = 8; i < n - (n % 8); i += 8)
        for (int j = 0; j < 8; ++j) r[j] += a[i + j];
    double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < n; ++i) res += a[i];
    return res;
}
// the recursion "n2 = n/2 - (n/2)%8; sum(a, n2) + sum(a+n2, n-n2)" unrolled onto an explicit stack (device
// recursion would need a run-time stack size)
__device__ double np_pairwise_sum(const double* a, int n) {
    struct Frame { int off, n, state; double left; };
    Frame st[32];
    int sp = 0;
    double ret = 0.0;
    st[sp++] = Frame{0, n, 0, 0.0};
    while (sp) {
        Frame& f = st[sp - 1];
        if (f.n <= 128) { ret = np_pairwise_leaf(a + f.off, f.n); --sp; continue; }
        int n2 = f.n / 2;
        n2 -= n2 % 8;
        if (f.state == 0) { f.state = 1; st[sp++] = Frame{f.off, n2, 0, 0.0}; continue; }
        if (f.state == 1) { f.left = ret; f.state = 2; st[sp++] = Frame{f.off + n2, f.n - n2, 0, 0.0}; continue; }
        ret = f.left + ret;
        --sp;
    }
    return ret;
}

// per-class bookkeeping of the multi-class evaluation (all NULL in the binary one)
struct ClassInfo {
    const int* ncomp_g; const int* ncomp_p;   // [N, C] components per class
    const int* ninst_g; const int* ninst_p;   // [N, C] instances (ids) per class; slot 0 includes id 0
};

// one warp per (tile, class): compact the PQ match IoUs of the class in gt-id order (== row-major order of
// np.nonzero), sum them the numpy way, and write the result records.
//   binary (ci.ncomp_g == NULL): class slot c0 = 1, records [N, 1]
//   multi-class: slots 0..C-1, records [N, C] with the branch rules of inst_metrics.py:103-131, 247-273
__global__ void k_metrics_final(InstState s, ClassInfo ci, const unsigned long long* IU, const int* tp,
                                double* scratch, int c0, int Cout, double* aji, double* pq) {
    int n = blockIdx.x, j = blockIdx.y, cls = c0 + j;
    int lane = threadIdx.x;
    long long o = (long long)n * s.KS;
    int ng = s.ng[n], np = s.np[n];
    bool multi = ci.ncomp_g != nullptr;
    // compaction slice: classes before this one own the first sum(ncomp_g[< cls]) entries
    int off = 0;
    if (multi) for (int t = 0; t < cls; ++t) off += ci.ncomp_g[n * s.C + t];
    double* buf = scratch + o + off;
    int m = 0;
    for (int base = 1; base <= ng; base += 32) {
        int gid = base + lane;
        double v = (gid <= ng && s.class_g(o, gid) == cls) ? s.pqiou[o + gid] : 0.0;
        unsigned b = __ballot_sync(0xffffffffu, v != 0.0);
        if (v != 0.0) buf[m + __popc(b & ((1u << lane) - 1))] = v;
        m += __popc(b);
    }
    __syncwarp();
    if (lane != 0) return;
    long long r = (long long)n * Cout + j;
    double I = (double)IU[((long long)n * s.C + cls) * 2], U = (double)IU[((long long)n * s.C + cls) * 2 + 1];
    int t = tp[n * s.C + cls];
    double iou = np_pairwise_sum(buf, m);
    if (!multi) {
        bool empty = ng == 0 || np == 0;                     // inst_metrics.py:72-73: (0., 0.) and nothing else
        if (aji) { aji[2 * r] = empty ? 0.0 : I; aji[2 * r + 1] = empty ? 0.0 : U; }
        if (pq) { pq[4 * r] = t; pq[4 * r + 1] = np - t; pq[4 * r + 2] = ng - t; pq[4 * r + 3] = iou; }
        return;
    }
    int ig = ci.ninst_g[n * s.C + cls], ip = ci.ninst_p[n * s.C + cls];
    int kg = ci.ncomp_g[n * s.C + cls], kp = ci.ncomp_p[n * s.C + cls];
    if (aji) { aji[2 * r] = I; aji[2 * r + 1] = U; }         // one-sided classes: all areas unpaired => same sums
    if (pq) {
        double vtp = 0, vfp = 0, vfn = 0, viou = 0;
        if (cls == 0) { vfp = ip; vfn = ig; }                                   // :249-252 (id 0 counted)
        else if (ip > 0 && ig > 0) { vtp = t; vfp = kp - t; vfn = kg - t; viou = iou; }   // :254-266
        else if (ip > 0) vfp = ip;                                              // :267-269 counts ids
        else if (ig > 0) vfn = ig;                                              // :270-272
        pq[4 * r] = vtp; pq[4 * r + 1] = vfp; pq[4 * r + 2] = vfn; pq[4 * r + 3] = viou;
    }
}

// ---- K13 semantic counts ---------------------------------------------------------------------------
// counts[n, k, c], k = TP, FP, FN, Pred, GT.  Each block keeps the (C+1) x (C+1) confusion matrix (gt, pred) of its
// pixels in shared memory — index C collects classes outside [0, C), which torch.histc does not count — with ONE
// shared atomic per group of lanes holding the same (gt, pred) pair (match_any), then derives the five vectors
// and flushes one global atomic per non-zero entry.
#define SEM_MAXC 64
__global__ void __launch_bounds__(TISEG_THREADS)
k_sem_counts(long long P, const uint8_t* __restrict__ pred, const uint8_t* __restrict__ gt, int C, int ignore,
             unsigned long long* counts, unsigned long long* valid, bool vec) {
    __shared__ unsigned h[(SEM_MAXC + 1) * (SEM_MAXC + 1)];
    const int C1 = C + 1, lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < C1 * C1; i += blockDim.x) h[i] = 0;
    __syncthreads();
    const long long base = (long long)blockIdx.y * P;
    // each thread walks several 4-pixel groups so that one block amortises its flush; the trip count is uniform
    const long long step = (long long)gridDim.x * blockDim.x * 4;
    if (C1 * C1 <= 16) {
        // few classes: every thread counts its own pixels (16 per trip, one 128-bit load per map) in 16 packed 8-bit
        // fields, flushed every 15 trips; the warp adds the fields up with redux and lane 0 posts them to the block
        // histogram
        unsigned long long a0 = 0ull, a1 = 0ull;
        int trips = 0;
        const bool vec16 = vec && (P % 16 == 0) && ((((uintptr_t)(pred + base)) | ((uintptr_t)(gt + base))) & 15) == 0;
        const long long step16 = (long long)gridDim.x * blockDim.x * 16;
        // all-vector case: four 128-bit loads per map in flight per thread (the pass is bound by bytes in flight)
        if (vec16) {
            // two classes, sixteen pixels whose bytes are all 0 / 1: the four words of each map fold into one (bit k of
            // byte j = pixel 4k + j) and the joint counts are three population counts
            const bool bin = C == 2 && ignore > 1;
            unsigned n11 = 0, n01 = 0, n10 = 0, n00 = 0;         // (gt, pred)
            const long long step64 = (long long)gridDim.x * blockDim.x * 64;
            for (long long i0 = (long long)blockIdx.x * blockDim.x * 64; i0 < P; i0 += step64) {
                uint4 a[4], b[4];
                int npx[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const long long i = i0 + ((long long)u * blockDim.x + threadIdx.x) * 16;
                    npx[u] = i < P ? 16 : 0;                     // (P % 16 == 0)
                    a[u] = make_uint4(0u, 0u, 0u, 0u); b[u] = a[u];
                    if (npx[u]) { a[u] = *reinterpret_cast<const uint4*>(pred + base + i); b[u] = *reinterpret_cast<const uint4*>(gt + base + i); }
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    if (npx[u] && bin && !((a[u].x | a[u].y | a[u].z | a[u].w | b[u].x | b[u].y | b[u].z | b[u].w) & 0xfefefefeu)) {
                        const unsigned pp = a[u].x | a[u].y << 1 | a[u].z << 2 | a[u].w << 3;
                        const unsigned tt = b[u].x | b[u].y << 1 | b[u].z << 2 | b[u].w << 3;
                        const unsigned c11 = __popc(pp & tt), cp = __popc(pp), ct = __popc(tt);
                        n11 += c11; n01 += cp - c11; n10 += ct - c11; n00 += 16u - cp - ct + c11;
                    } else
                    if (npx[u]) {
                        const unsigned pw[4] = {a[u].x, a[u].y, a[u].z, a[u].w}, tw[4] = {b[u].x, b[u].y, b[u].z, b[u].w};
#pragma unroll
                        for (int k = 0; k < 16; ++k) {
                            const int p = (pw[k >> 2] >> (8 * (k & 3))) & 255, t = (tw[k >> 2] >> (8 * (k & 3))) & 255;
                            if (t != ignore) {
                                const int key = min(t, C) * C1 + min(p, C);
                                const unsigned long long one = 1ull << ((key & 7) * 8);
                                if (key < 8) a0 += one; else a1 += one;
                            }
                        }
                    }
                    if (++trips == 15 || (u == 3 && i0 + step64 >= P)) {
#pragma unroll
                        for (int key = 0; key < 16; ++key) {
                            const unsigned f = (unsigned)(((key < 8 ? a0 : a1) >> ((key & 7) * 8)) & 0xffull);
                            const unsigned tot = __reduce_add_sync(0xffffffffu, f);
                            if (lane == 0 && tot && key < C1 * C1) atomicAdd(&h[key], tot);
                        }
                        a0 = a1 = 0ull; trips = 0;
                    }
                }
            }
            if (bin) {                                           // (uniform; C1 = 3: key = gt * 3 + pred)
                n00 = __reduce_add_sync(0xffffffffu, n00); n01 = __reduce_add_sync(0xffffffffu, n01);
                n10 = __reduce_add_sync(0xffffffffu, n10); n11 = __reduce_add_sync(0xffffffffu, n11);
                if (lane == 0) {
                    if (n00) atomicAdd(&h[0], n00);
                    if (n01) atomicAdd(&h[1], n01);
                    if (n10) atomicAdd(&h[3], n10);
                    if (n11) atomicAdd(&h[4], n11);
                }
            }
        } else
        for (long long i0 = (long long)blockIdx.x * blockDim.x * 16; i0 < P; i0 += step16) {
            const long long i = i0 + (long long)threadIdx.x * 16;
            unsigned pw[4] = {0u, 0u, 0u, 0u}, tw[4] = {0u, 0u, 0u, 0u};
            int npx = 0;
            if (i < P) {
                npx = (int)(P - i < 16 ? P - i : 16);
                if (vec16) {
                    const uint4 a = *reinterpret_cast<const uint4*>(pred + base + i), b = *reinterpret_cast<const uint4*>(gt + base + i);
                    pw[0] = a.x; pw[1] = a.y; pw[2] = a.z; pw[3] = a.w;
                    tw[0] = b.x; tw[1] = b.y; tw[2] = b.z; tw[3] = b.w;
                } else {
#pragma unroll
                    for (int k = 0; k < 16; ++k) {               // (unrolled: pw / tw stay in registers)
                        if (k < npx) {
                            pw[k >> 2] |= (unsigned)pred[base + i + k] << (8 * (k & 3));
                            tw[k >> 2] |= (unsigned)gt[base + i + k] << (8 * (k & 3));
                        }
                    }
                }
            }
#pragma unroll
            for (int k = 0; k < 16; ++k) {
                if (k < npx) {
                    const int p = (pw[k >> 2] >> (8 * (k & 3))) & 255, t = (tw[k >> 2] >> (8 * (k & 3))) & 255;
                    if (t != ignore) {
                        const int key = min(t, C) * C1 + min(p, C);
                        const unsigned long long one = 1ull << ((key & 7) * 8);
                        if (key < 8) a0 += one; else a1 += one;
                    }
                }
            }
            if (++trips == 15 || i0 + step16 >= P) {
#pragma unroll
                for (int key = 0; key < 16; ++key) {
                    const unsigned f = (unsigned)(((key < 8 ? a0 : a1) >> ((key & 7) * 8)) & 0xffull);
                    const unsigned tot = __reduce_add_sync(0xffffffffu, f);
                    if (lane == 0 && tot && key < C1 * C1) atomicAdd(&h[key], tot);
                }
                a0 = a1 = 0ull; trips = 0;
            }
        }
    } else
    for (long long i0 = (long long)blockIdx.x * blockDim.x * 4; i0 < P; i0 += step) {
        const long long i = i0 + (long long)threadIdx.x * 4;
        Pack4<uint8_t> pp, tt;
        if (i < P) { pp = ld4(pred + base, i, P, vec); tt = ld4(gt + base, i, P, vec); }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            int key = -1;
            if (i + k < P) {
                const int p = pp.v[k], t = tt.v[k];
                if (t != ignore) key = min(t, C) * C1 + min(p, C);
            }
            const unsigned peers = __match_any_sync(0xffffffffu, key);
            if (key >= 0 && lane == __ffs(peers) - 1) atomicAdd(&h[key], (unsigned)__popc(peers));
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 5 * C; i += blockDim.x) {
        const int k = i / C, c = i - k * C;
        unsigned v = 0;
        if (k == 0) v = h[c * C1 + c];
        else if (k == 1) { for (int t = 0; t <= C; ++t) if (t != c) v += h[t * C1 + c]; }
        else if (k == 2) { for (int q = 0; q <= C; ++q) if (q != c) v += h[c * C1 + q]; }
        else if (k == 3) { for (int t = 0; t <= C; ++t) v += h[t * C1 + c]; }
        else { for (int q = 0; q <= C; ++q) v += h[c * C1 + q]; }
        if (v) atomicAdd(&counts[(long long)blockIdx.y * 5 * C + i], (unsigned long long)v);
    }
    if (threadIdx.x < 32) {
        unsigned nv = 0;
        for (int i = lane; i < C1 * C1; i += 32) nv += h[i];
        for (int d = 16; d; d >>= 1) nv += __shfl_down_sync(0xffffffffu, nv, d);
        if (lane == 0 && nv) atomicAdd(&valid[blockIdx.y], (unsigned long long)nv);
    }
}

static int next_pow2(long long v) { int p = 1; while (p < v) p <<= 1; return p; }

// ---- instance -> class assignment (assign_sem_class_to_insts, datasets/utils/instance_semantic.py:68-93) ----
// hist[n, v, 0..C] = pixels of instance value v per semantic class (slot C collects out-of-range classes so
// that the instance still exists); one atomic per in-segment run of equal (instance, class)
__global__ void __launch_bounds__(TISEG_THREADS)
k_inst_class_hist(Geom g, const int32_t* __restrict__ inst, const uint8_t* __restrict__ sem, int C, int VM,
                  int* hist, int* bad) {
    Pix px;
    if (!warp_pixel(g, px)) return;
    int v = 0, c = 0;
    if (px.ok) { v = inst[px.base + px.idx]; c = sem[px.base + px.idx]; if (c >= C) c = C; }
    int key = v * (C + 1) + c;
    int kl = __shfl_up_sync(0xffffffffu, key, 1);
    bool cont = px.lane > 0 && key == kl;
    unsigned m = __ballot_sync(0xffffffffu, cont);
    if (px.ok && v != 0 && !cont) {
        if (v < 0 || v >= VM) { *bad = 1; return; }
        atomicAdd(&hist[((long long)px.n * VM + v) * (C + 1) + c], run_end_lane(m, px.lane) - px.lane + 1);
    }
}

// The class tables are addressed by instance id with a stride of VM = max(P + 1, 65536) entries per tile, but only the ids
// that occur can be touched: the largest id of every tile is found first, and clearing / scanning stop there (a CoNIC
// batch of 512 tiles has ~60 instances each: 1 GB of table shrinks to a few hundred KB of traffic).
__global__ void __launch_bounds__(TISEG_THREADS) k_max_id(Geom g, const int32_t* __restrict__ inst, int* __restrict__ maxid) {
    const int n = blockIdx.y;
    const int32_t* t = inst + (long long)n * g.P;
    int m = 0;
    for (long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4; i < g.P; i += (long long)gridDim.x * blockDim.x * 4) {
        if (i + 3 < g.P && ((((uintptr_t)t) | (g.P * 4ull)) & 15) == 0) { const int4 q = *reinterpret_cast<const int4*>(t + i); m = max(max(m, max(q.x, q.y)), max(q.z, q.w)); }
        else for (int k = 0; k < 4 && i + k < g.P; ++k) m = max(m, t[i + k]);
    }
    m = __reduce_max_sync(0xffffffffu, m);
    if ((threadIdx.x & 31) == 0 && m > 0) atomicMax(&maxid[n], m);
}
__global__ void k_zero_class_hist(int* __restrict__ hist, int C, int VM, const int* __restrict__ maxid) {
    const int n = blockIdx.y;
    const long long top = (long long)min(maxid[n], VM - 1) * (C + 1) + C;              // last entry that can be touched
    int* h = hist + (long long)n * VM * (C + 1);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i <= top; i += (long long)gridDim.x * blockDim.x) h[i] = 0;
}

__global__ void k_inst_class_pick(const int* __restrict__ hist, int C, int VM, uint8_t* cls_inst, int* ninst, const int* __restrict__ maxid) {
    int n = blockIdx.y;
    const int top = min(maxid[n], VM - 1);
    for (int v = blockIdx.x * blockDim.x + threadIdx.x; v <= top; v += gridDim.x * blockDim.x) {
    int cls = -1;
    if (v == 0) cls = 0;                                     // id 0 is always listed under class 0
    else {
        const int* h = hist + ((long long)n * VM + v) * (C + 1);
        int tot = 0, best = 0, bc = 0, fg = 0;
        for (int c = 0; c <= C; ++c) tot += h[c];
        if (tot > 0) {
            for (int c = 1; c < C; ++c) { fg += h[c]; if (h[c] > best) { best = h[c]; bc = c; } }   // first max
            cls = fg > 0 ? bc : 0;
        }
    }
    if (cls >= 0) { cls_inst[(long long)n * VM + v] = (uint8_t)cls; atomicAdd(&ninst[n * C + cls], 1); }
    }
}

// class of every connected component = class of the instance value at its root pixel (from the bitmap of the roots)
__global__ void __launch_bounds__(TISEG_THREADS)
k_comp_class_bits(Geom g, const int32_t* __restrict__ inst, const unsigned* __restrict__ rootbits, const int* __restrict__ rank,
                  const uint8_t* __restrict__ cls_inst, int VM, int C, uint8_t* cls_comp, int KS, int* ncomp) {
    const long long words = (long long)g.H * g.SEG;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= words) return;
    const int n = blockIdx.y;
    unsigned m = rootbits[(long long)n * words + t];
    if (!m) return;
    const int y = (int)(t / g.SEG), seg = (int)(t - (long long)y * g.SEG);
    const long long base = (long long)n * g.P;
    while (m) {
        const int b = __ffs(m) - 1;
        m &= m - 1;
        const int idx = y * g.W + seg * 32 + b;
        const int v = inst[base + idx];
        const int cls = (v > 0 && v < VM) ? cls_inst[(long long)n * VM + v] : 0;
        cls_comp[(long long)n * KS + rank[base + idx]] = (uint8_t)cls;
        atomicAdd(&ncomp[n * C + cls], 1);
    }
}

struct PairWork {              // everything one evaluation shares: forests, ids, areas, the pair table
    InstState s;
    PairTab t;
    double* scratch;
};

// Roots of the two labellings: rank (raster-order id) valid at the root pixels, and the bitmap of the roots.
struct PairRoots {
    const int* rank_g; const int* rank_p;
    const unsigned* bits_g; const unsigned* bits_p;
};

static int pair_state_alloc(tiseg_ctx* c, const Geom& g, PairWork& w, int** ng, int** np, int** overflow) {
    const int N = g.N, KS = g.P + 1;
    const size_t ks = (size_t)N * KS;
    InstState& s = w.s;
    *ng = ws<int>(c, (size_t)2 * N); *np = *ng ? *ng + N : nullptr;       // contiguous: pair_table_build ranks 2N tiles at once
    s.area_g = ws<int>(c, ks); s.area_p = ws<int>(c, ks);
    s.best = ws<unsigned long long>(c, ks); s.bestp = ws<int>(c, ks);
    s.used = ws<uint8_t>(c, ks); s.pqiou = ws<double>(c, ks);
    w.scratch = ws<double>(c, ks);
    *overflow = ws<int>(c, 1);
    if (!*ng || !s.area_g || !s.area_p || !s.best || !s.bestp || !s.used || !s.pqiou || !w.scratch || !*overflow) return TISEG_ERR_CUDA;
    s.ng = *ng; s.np = *np; s.KS = KS; s.cls_g = nullptr; s.cls_p = nullptr; s.C = 2;
    return TISEG_OK;
}

static int pair_tab_alloc(tiseg_ctx* c, const Geom& g, PairTab& t, int* overflow) {
    const int N = g.N;
    t.small.cap = next_pow2(g.P / 32 < 1024 ? 1024 : g.P / 32);
    t.big.cap = next_pow2(2ll * g.P);
    t.small.key = ws<unsigned long long>(c, (size_t)N * t.small.cap);
    t.small.cnt = ws<int>(c, (size_t)N * t.small.cap);
    t.big.key = ws<unsigned long long>(c, (size_t)N * t.big.cap);
    t.big.cnt = ws<int>(c, (size_t)N * t.big.cap);
    t.overflow = overflow;
    if (!t.small.key || !t.small.cnt || !t.big.key || !t.big.cnt) return TISEG_ERR_CUDA;
    const size_t kb = (size_t)N * t.small.cap * sizeof(unsigned long long), cb = (size_t)N * t.small.cap * sizeof(int);
    if ((char*)t.small.cnt == (char*)t.small.key + kb) return zero(c, t.small.key, kb + cb);     // adjacent: one memset
    TISEG_TRY(zero(c, t.small.key, kb));
    return zero(c, t.small.cnt, cb);
}

// from bit planes (see the comment above k_pair_bits)
static int pair_table_build(tiseg_ctx* c, const Geom& g, const int32_t* d_pred, const int32_t* d_gt, PairWork& w,
                            PairRoots* roots, const uint16_t* d_gt16 = nullptr) {
    const int N = g.N;
    const size_t total = (size_t)N * g.P, words = (size_t)N * g.H * g.SEG;
    BitPlanesW pw;
    TISEG_TRY(bitplanes_alloc(c, g, 2, pw));
    int* par = ws<int>(c, 2 * total);
    int* rank = ws<int>(c, 2 * total);
    unsigned* lbits = ws<unsigned>(c, 2 * words);
    unsigned* fbits = ws<unsigned>(c, 2 * words);
    int *ng, *np, *overflow;
    if (!par || !rank || !lbits || !fbits) return TISEG_ERR_CUDA;
    TISEG_TRY(pair_state_alloc(c, g, w, &ng, &np, &overflow));
    InstState& s = w.s;
    PairTab& t = w.t;
    TISEG_TRY(pair_tab_alloc(c, g, t, overflow));
    TISEG_TRY(zero(c, overflow, sizeof(int)));
    // measure.label(inst.copy()) on both maps (inst_metrics.py:12-13): equal-value, 8-connected, background 0
    const long long warps = (long long)((g.W + 255) / 256) * ((g.H + EQ_BAND - 1) / EQ_BAND);
    const dim3 eg((unsigned)((warps + TISEG_WARPS_PER_BLOCK - 1) / TISEG_WARPS_PER_BLOCK), (unsigned)N);
    BitPlanesW pwp = {pw.F + words, pw.C + words, pw.EU + words, pw.EL + words, pw.ER + words};
    if (d_gt16) TISEG_LAUNCH(c, k_eqbits<uint16_t>, eg, TISEG_THREADS, 0, g, d_gt16, pw, (g.W % 4 == 0) && (((uintptr_t)d_gt16) & 7) == 0);
    else TISEG_LAUNCH(c, k_eqbits<int32_t>, eg, TISEG_THREADS, 0, g, d_gt, pw, (g.W % 4 == 0) && aligned16(d_gt));
    TISEG_LAUNCH(c, k_eqbits<int32_t>, eg, TISEG_THREADS, 0, g, d_pred, pwp, (g.W % 4 == 0) && aligned16(d_pred));
    const BitPlanes p = as_const(pw);
    Geom g2 = make_geom(2 * N, g.H, g.W);                  // both maps as one batch: gt tiles, then pred tiles
    TISEG_TRY(bitccl_build(c, g2, p, 2, par, lbits, fbits));
    TISEG_TRY(rank_from_bits(c, g2, fbits, rank, ng));     // counts: ng[0..N) then np[0..N)
    TISEG_LAUNCH(c, k_inst_init, dim3(16, N), 256, 0, s, 1);
    const dim3 wgrid((unsigned)(((long long)g.H * g.SEG + TISEG_THREADS - 1) / TISEG_THREADS), (unsigned)N);
    TISEG_LAUNCH(c, k_pair_bits<false>, wgrid, TISEG_THREADS, 0, g, p, par, rank, s, t, c->d_err + 1);
    // a pathological input overflowed the small table: clear the always-sufficient one and redo (idle otherwise)
    TISEG_LAUNCH(c, k_pair_zero_big, c->sm_count * 8, TISEG_THREADS, 0, t, t, N);
    TISEG_LAUNCH(c, k_pair_bits<true>, wgrid, TISEG_THREADS, 0, g, p, par, rank, s, t, c->d_err + 1);
    if (roots) *roots = PairRoots{rank, rank + total, fbits, fbits + words};
    return TISEG_OK;
}

// AJI / PQ records from a built table; cls_* NULL = binary
static int pair_eval(tiseg_ctx* c, const Geom& g, PairWork& w, const uint8_t* cls_g, const uint8_t* cls_p, int C,
                     const ClassInfo& ci, bool first_eval, double* d_aji, double* d_pq, double match_iou = 0.5) {
    int N = g.N;
    InstState s = w.s;
    s.cls_g = cls_g; s.cls_p = cls_p; s.C = C;
    unsigned long long* IU = ws<unsigned long long>(c, 2 * (size_t)N * C);
    int* tp = ws<int>(c, (size_t)N * C);
    if (!IU || !tp) return TISEG_ERR_CUDA;
    TISEG_TRY(zero(c, IU, 2 * (size_t)N * C * sizeof(unsigned long long)));
    TISEG_TRY(zero(c, tp, (size_t)N * C * sizeof(int)));
    if (!first_eval) TISEG_LAUNCH(c, k_inst_init, dim3(16, N), 256, 0, s, 0);
    dim3 tg((w.t.small.cap + 255) / 256, N);                 // the kernels stride over the table in force
    TISEG_LAUNCH(c, k_pair_best, tg, 256, 0, w.t, s, tp, match_iou);
    TISEG_LAUNCH(c, k_pair_argbest, tg, 256, 0, w.t, s);
    TISEG_LAUNCH(c, k_aji_gt, dim3(8, N), 256, 0, w.t, s, IU);
    TISEG_LAUNCH(c, k_aji_pred, dim3(8, N), 256, 0, s, IU);
    bool multi = cls_g != nullptr;
    TISEG_LAUNCH(c, k_metrics_final, dim3(N, multi ? C : 1), 32, 0, s, ci, IU, tp, w.scratch, multi ? 0 : 1,
                 multi ? C : 1, d_aji, d_pq);
    return TISEG_OK;
}

// class of every component of one side (pred or gt)
static int side_classes(tiseg_ctx* c, const Geom& g, const int32_t* inst, const uint8_t* sem, const int* rank,
                        const unsigned* rootbits, int C, int VM, uint8_t** cls_comp_out, int** ncomp_out, int** ninst_out,
                        int* bad) {
    int N = g.N, KS = g.P + 1;
    int* hist = ws<int>(c, (size_t)N * VM * (C + 1));
    uint8_t* cls_inst = ws<uint8_t>(c, (size_t)N * VM);
    uint8_t* cls_comp = ws<uint8_t>(c, (size_t)N * KS);
    int* ncomp = ws<int>(c, (size_t)N * C);
    int* ninst = ws<int>(c, (size_t)N * C);
    int* maxid = ws<int>(c, (size_t)N);
    if (!hist || !cls_inst || !cls_comp || !ncomp || !ninst || !maxid) return TISEG_ERR_CUDA;
    TISEG_TRY(zero(c, ncomp, (size_t)N * C * sizeof(int)));
    TISEG_TRY(zero(c, ninst, (size_t)N * C * sizeof(int)));
    TISEG_TRY(zero(c, maxid, (size_t)N * sizeof(int)));
    TISEG_LAUNCH(c, k_max_id, dim3(8, N), TISEG_THREADS, 0, g, inst, maxid);
    TISEG_LAUNCH(c, k_zero_class_hist, dim3(8, N), 256, 0, hist, C, VM, maxid);
    TISEG_LAUNCH(c, k_inst_class_hist, warp_grid(g), TISEG_THREADS, 0, g, inst, sem, C, VM, hist, bad);
    TISEG_LAUNCH(c, k_inst_class_pick, dim3(8, N), 256, 0, hist, C, VM, cls_inst, ninst, maxid);
    TISEG_LAUNCH(c, k_comp_class_bits, dim3((unsigned)(((long long)g.H * g.SEG + TISEG_THREADS - 1) / TISEG_THREADS), (unsigned)N),
                 TISEG_THREADS, 0, g, inst, rootbits, rank, cls_inst, VM, C, cls_comp, KS, ncomp);
    *cls_comp_out = cls_comp; *ncomp_out = ncomp; *ninst_out = ninst;
    return TISEG_OK;
}

}  // namespace tiseg

using namespace tiseg;

// cls_out[n, v] = semantic class of instance id v (first argmax over classes >= 1, 0 without a non-background pixel), 255 = no such id
__global__ void k_inst_class_table(const int* __restrict__ hist, int C, int VM, uint8_t* __restrict__ table) {
    int n = blockIdx.y;
    int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= VM) return;
    int cls = 255;
    if (v == 0) cls = 0;
    else {
        const int* h = hist + ((long long)n * VM + v) * (C + 1);
        int tot = 0, best = 0, bc = 0, fg = 0;
        for (int c = 0; c <= C; ++c) tot += h[c];
        if (tot > 0) {
            for (int c = 1; c < C; ++c) { fg += h[c]; if (h[c] > best) { best = h[c]; bc = c; } }
            cls = fg > 0 ? bc : 0;
        }
    }
    table[(long long)n * VM + v] = (uint8_t)cls;
}

extern "C" {

int tiseg_assign_sem_class(tiseg_ctx* c, const int32_t* inst, const uint8_t* sem, int N, int H, int W, int C, uint8_t* table_out) {
    if (!c || !inst || !sem || !table_out || C < 2 || C > 64) { set_error("tiseg_assign_sem_class: bad argument (2 <= C <= 64)"); return TISEG_ERR_ARG; }
    TISEG_TRY(check_geom(N, H, W));
    begin_call(c);
    Geom g = make_geom(N, H, W);
    size_t total = (size_t)N * g.P;
    const int VM = g.P + 1 < (1 << 16) ? (1 << 16) : g.P + 1;
    const int32_t* d_inst = in(c, inst, total);
    const uint8_t* d_sem = in(c, sem, total);
    uint8_t* d_tab = tiseg::out(c, table_out, (size_t)N * VM);
    int* hist = ws<int>(c, (size_t)N * VM * (C + 1));
    if (!d_inst || !d_sem || !d_tab || !hist) return TISEG_ERR_CUDA;
    TISEG_TRY(zero(c, hist, (size_t)N * VM * (C + 1) * sizeof(int)));
    TISEG_LAUNCH(c, k_inst_class_hist, warp_grid(g), TISEG_THREADS, 0, g, d_inst, d_sem, C, VM, hist, c->d_err);
    TISEG_LAUNCH(c, k_inst_class_table, dim3((VM + 255) / 256, N), 256, 0, hist, C, VM, d_tab);
    return end_call(c);
}

int tiseg_pair_metrics_bin(tiseg_ctx* c, const int32_t* pred, const int32_t* gt, int N, int H, int W,
                           double* aji, double* pq) {
    return tiseg_pair_metrics_bin_iou(c, pred, gt, N, H, W, 0.5, aji, pq);
}

static int pair_metrics_bin_any(tiseg_ctx* c, const int32_t* pred, const int32_t* gt, const uint16_t* gt16, int N, int H, int W,
                                double match_iou, double* aji, double* pq);

int tiseg_pair_metrics_bin_iou(tiseg_ctx* c, const int32_t* pred, const int32_t* gt, int N, int H, int W, double match_iou,
                               double* aji, double* pq) {
    return pair_metrics_bin_any(c, pred, gt, nullptr, N, H, W, match_iou, aji, pq);
}

int tiseg_pair_metrics_bin_u16gt(tiseg_ctx* c, const int32_t* pred, const uint16_t* gt, int N, int H, int W, double match_iou,
                                 double* aji, double* pq) {
    return pair_metrics_bin_any(c, pred, nullptr, gt, N, H, W, match_iou, aji, pq);
}

static int pair_metrics_bin_any(tiseg_ctx* c, const int32_t* pred, const int32_t* gt, const uint16_t* gt16, int N, int H, int W,
                                double match_iou, double* aji, double* pq) {
    if (!c || !pred || (!gt && !gt16) || !(match_iou >= 0.5)) {
        set_error("tiseg_pair_metrics_bin: bad argument (match_iou >= 0.5: below it the reference switches to Hungarian matching)");
        return TISEG_ERR_ARG;
    }
    TISEG_TRY(check_geom(N, H, W));
    begin_call(c);
    Geom g = make_geom(N, H, W);
    size_t total = (size_t)N * g.P;
    const int32_t* d_pred = in(c, pred, total);
    const int32_t* d_gt = gt ? in(c, gt, total) : nullptr;
    const uint16_t* d_gt16 = gt16 ? in(c, gt16, total) : nullptr;
    double* d_aji = aji ? tiseg::out(c, aji, 2 * (size_t)N) : nullptr;
    double* d_pq = pq ? tiseg::out(c, pq, 4 * (size_t)N) : nullptr;
    if (!d_pred || (!d_gt && !d_gt16)) return TISEG_ERR_CUDA;
    PairWork w;
    TISEG_TRY(pair_table_build(c, g, d_pred, d_gt, w, nullptr, d_gt16));
    ClassInfo ci = {nullptr, nullptr, nullptr, nullptr};
    TISEG_TRY(pair_eval(c, g, w, nullptr, nullptr, 2, ci, true, d_aji, d_pq, match_iou));
    return end_call(c);
}

int tiseg_pair_metrics_multiclass(tiseg_ctx* c, const int32_t* pred_inst, const uint8_t* pred_sem,
                                  const int32_t* gt_inst, const uint8_t* gt_sem, int N, int H, int W, int C,
                                  double* aji, double* pq, double* bin_aji, double* bin_pq) {
    if (!c || !pred_inst || !pred_sem || !gt_inst || !gt_sem || C < 2 || C > 64) {
        set_error("tiseg_pair_metrics_multiclass: bad argument (2 <= C <= 64)");
        return TISEG_ERR_ARG;
    }
    TISEG_TRY(check_geom(N, H, W));
    begin_call(c);
    Geom g = make_geom(N, H, W);
    size_t total = (size_t)N * g.P;
    const int32_t* d_pi = in(c, pred_inst, total);
    const uint8_t* d_ps = in(c, pred_sem, total);
    const int32_t* d_gi = in(c, gt_inst, total);
    const uint8_t* d_gs = in(c, gt_sem, total);
    double* d_aji = aji ? tiseg::out(c, aji, 2 * (size_t)N * C) : nullptr;
    double* d_pq = pq ? tiseg::out(c, pq, 4 * (size_t)N * C) : nullptr;
    double* d_baji = bin_aji ? tiseg::out(c, bin_aji, 2 * (size_t)N) : nullptr;
    double* d_bpq = bin_pq ? tiseg::out(c, bin_pq, 4 * (size_t)N) : nullptr;
    if (!d_pi || !d_ps || !d_gi || !d_gs) return TISEG_ERR_CUDA;
    PairWork w;
    PairRoots rt;
    TISEG_TRY(pair_table_build(c, g, d_pi, d_gi, w, &rt));
    ClassInfo none = {nullptr, nullptr, nullptr, nullptr};
    bool first = true;
    if (d_baji || d_bpq) { TISEG_TRY(pair_eval(c, g, w, nullptr, nullptr, 2, none, first, d_baji, d_bpq)); first = false; }
    if (d_aji || d_pq) {
        int VM = g.P + 1 < (1 << 16) ? (1 << 16) : g.P + 1;     // instance ids index the class tables directly
        int* bad = c->d_err;                                    // deferred: reported by the next synchronising call
        uint8_t *cls_g, *cls_p;
        ClassInfo ci;
        int *a, *b;
        TISEG_TRY(side_classes(c, g, d_gi, d_gs, rt.rank_g, rt.bits_g, C, VM, &cls_g, &a, &b, bad));
        ci.ncomp_g = a; ci.ninst_g = b;
        TISEG_TRY(side_classes(c, g, d_pi, d_ps, rt.rank_p, rt.bits_p, C, VM, &cls_p, &a, &b, bad));
        ci.ncomp_p = a; ci.ninst_p = b;
        TISEG_TRY(pair_eval(c, g, w, cls_g, cls_p, C, ci, first, d_aji, d_pq));
    }
    return end_call(c);
}

int tiseg_sem_counts(tiseg_ctx* c, const uint8_t* pred, const uint8_t* gt, int N, int H, int W, int C,
                     int ignore_index, int64_t* counts, int64_t* valid) {
    if (!c || !pred || !gt || !counts || !valid || C <= 0 || C > SEM_MAXC) { set_error("tiseg_sem_counts: bad argument (C <= 64)"); return TISEG_ERR_ARG; }
    TISEG_TRY(check_geom(N, H, W));
    begin_call(c);
    Geom g = make_geom(N, H, W);
    size_t total = (size_t)N * g.P;
    const uint8_t* d_pred = in(c, pred, total);
    const uint8_t* d_gt = in(c, gt, total);
    int64_t* d_counts = tiseg::out(c, counts, (size_t)N * 5 * C);
    int64_t* d_valid = tiseg::out(c, valid, (size_t)N);
    if (!d_pred || !d_gt || !d_counts || !d_valid) return TISEG_ERR_CUDA;
    TISEG_TRY(zero(c, d_counts, (size_t)N * 5 * C * sizeof(int64_t)));
    TISEG_TRY(zero(c, d_valid, (size_t)N * sizeof(int64_t)));
    unsigned gx = flat4_grid(g.P);
    gx = gx > 64 ? (gx + 7) / 8 : gx;                         // ~8 groups per thread
    // the 16-pixel path: few blocks per tile with many trips each — every block ends with 5C + 1 global atomics on the
    // handful of cache lines that hold the counters, and those serialise in L2
    if ((C + 1) * (C + 1) <= 16 && gx > 16) gx = 16;
    if ((C + 1) * (C + 1) <= 16 && (long long)N * gx < 4ll * c->sm_count) {          // few tiles: more blocks per tile
        const long long want = (4ll * c->sm_count + N - 1) / N, most = ((long long)g.P + 64 * TISEG_THREADS - 1) / (64 * TISEG_THREADS);
        gx = (unsigned)(want < most ? want : most);
        if (gx < 1) gx = 1;
    }
    bool vec = (g.P % 4 == 0) && ((((uintptr_t)d_pred) | ((uintptr_t)d_gt)) & 3) == 0;
    TISEG_LAUNCH(c, k_sem_counts, dim3(gx, N), TISEG_THREADS, 0, (long long)g.P, d_pred, d_gt, C, ignore_index,
                 (unsigned long long*)d_counts, (unsigned long long*)d_valid, vec);
    return end_call(c);
}

}  // extern "C"
