// tiseg_b200 — shared device/host plumbing for the sm_100a kernels of the test-time instance pipeline.
//
// Layout convention (every kernel): a BATCH of tiles [N, H, W], C-contiguous, row pitch = W elements.
// Class maps / masks are uint8, label maps int32, float maps fp32 / fp64.  One warp owns a 32-pixel
// horizontal segment of one row (coalesced 128-byte int32 or 32-byte uint8 requests); the warp-level
// run primitives (ballot / clz) below are what the CCL, histogram and area kernels build on.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>

#include "../../include/tiseg_b200.h"

#define TISEG_WARPS_PER_BLOCK 8
#define TISEG_THREADS (32 * TISEG_WARPS_PER_BLOCK)

struct tiseg_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaEvent_t order_ev = nullptr;   // orders a newly bound stream after the work queued on the previous one
    // device arena: list of blocks, bump-allocated per call, coalesced between calls
    struct Block { char* p; size_t cap; };
    std::vector<Block> blocks;
    size_t cur_block = 0, cur_off = 0, call_total = 0;
    // pending device->host copies of the current call
    struct Pending { void* host; const void* dev; size_t bytes; };
    std::vector<Pending> pending;
    long long launches = 0;
    int sm_count = 148;
    // data-dependent errors raised by kernels (word 0: instance id out of range, word 1: internal table loss).  A
    // call that synchronises anyway (host outputs) reports them itself; stream-ordered calls with device outputs
    // return before execution and leave them to the next call that synchronises (tiseg_synchronize included).
    int* d_err = nullptr;      // [2] device
    int* h_err = nullptr;      // [2] pinned host mirror
    // dynamic shared-memory limits of the flood kernels, raised once on this context's device (cudaFuncSetAttribute acts
    // on the current device, so the flag belongs with the device and not with the process)
    bool smem_flood_u8[2] = {false, false};    // k_ws_flood_par<false>, k_ws_flood_par<true>
    bool smem_flood_f64 = false;               // k_rank_blobs<true>, k_ws_flood_ranked
    // optional per-kernel CUDA-event timing (bench.py's roofline leg); off by default
    bool timing = false;
    struct Timed { const char* name; cudaEvent_t a, b; };
    std::vector<Timed> timed;
    std::vector<cudaEvent_t> event_pool;
};

namespace tiseg {

void set_error(const std::string& msg);
int fail(const char* where, cudaError_t e);

// ---- call-scoped workspace -------------------------------------------------------------------
int check_deferred(tiseg_ctx* c);                 // after a stream sync: report + clear kernel-raised errors
void* ws_alloc(tiseg_ctx* c, size_t bytes);       // 256-byte aligned device scratch, valid until the next call

template <class T> inline T* ws(tiseg_ctx* c, size_t n) { return (T*)ws_alloc(c, n * sizeof(T)); }

int zero(tiseg_ctx* c, void* p, size_t bytes);
// records the 'before' event of a timed launch and returns the 'after' event to record
cudaEvent_t timing_before(tiseg_ctx* c, const char* name);

#define TISEG_CHECK(expr)                                                \
    do {                                                                 \
        cudaError_t _e = (expr);                                         \
        if (_e != cudaSuccess) return ::tiseg::fail(#expr, _e);          \
    } while (0)

#define TISEG_TRY(expr)                 \
    do {                                \
        int _s = (expr);                \
        if (_s != TISEG_OK) return _s;  \
    } while (0)

// launch + count + error check.  Usage: TISEG_LAUNCH(c, kernel, grid, block, smem, args...)
#define TISEG_LAUNCH_AS(c, name, kern, grid, block, smem, ...)                        \
    do {                                                                              \
        cudaEvent_t _tb = (c)->timing ? ::tiseg::timing_before((c), name) : nullptr;  \
        kern<<<(grid), (block), (smem), (c)->stream>>>(__VA_ARGS__);                  \
        if (_tb) cudaEventRecord(_tb, (c)->stream);                                   \
        (c)->launches++;                                                              \
        cudaError_t _e = cudaGetLastError();                                          \
        if (_e != cudaSuccess) return ::tiseg::fail(name, _e);                        \
    } while (0)
#define TISEG_LAUNCH(c, kern, grid, block, smem, ...) TISEG_LAUNCH_AS(c, #kern, kern, grid, block, smem, __VA_ARGS__)

// ---- geometry: one warp per 32-pixel row segment, blocks never straddle two tiles ----------------
struct Geom {
    int N, H, W, SEG;          // SEG = ceil(W / 32)
    int P;                     // H * W  (< 2^31: tile-local flat indices are int)
    int wpt;                   // warps per tile = H * SEG
    int bpt;                   // blocks per tile = ceil(wpt / 8)
    // "listed" mode (kernels written with FOR_TILES): the launch has ONE tile slot (gridDim.y = 1) and every block
    // loops over the device-side list tl[0 .. *tn) — normally empty, so a rarely needed general path costs a few
    // microseconds of empty blocks instead of a host round trip to decide whether to launch it.
    const int* tl;
    const int* tn;
};
inline Geom make_geom(int N, int H, int W) {
    Geom g; g.N = N; g.H = H; g.W = W; g.SEG = (W + 31) / 32; g.P = H * W;
    g.wpt = H * g.SEG; g.bpt = (g.wpt + TISEG_WARPS_PER_BLOCK - 1) / TISEG_WARPS_PER_BLOCK;
    g.tl = nullptr; g.tn = nullptr; return g;
}
inline Geom listed_geom(Geom g, const int* list, const int* count) { g.tl = list; g.tn = count; return g; }
inline unsigned grid_tiles(const Geom& g) { return g.tl ? 1u : (unsigned)g.N; }
inline dim3 warp_grid(const Geom& g) { return dim3((unsigned)g.bpt, grid_tiles(g), 1); }
inline unsigned flat_grid(long long n, int per_block = TISEG_THREADS) { return (unsigned)((n + per_block - 1) / per_block); }
inline unsigned flat4_grid(long long n) { return (unsigned)((n + 4 * TISEG_THREADS - 1) / (4 * TISEG_THREADS)); }
inline bool aligned16(const void* a, const void* b = nullptr, const void* c = nullptr, const void* d = nullptr, const void* e = nullptr) {
    return ((((uintptr_t)a) | ((uintptr_t)b) | ((uintptr_t)c) | ((uintptr_t)d) | ((uintptr_t)e)) & 15) == 0;
}
inline int check_geom(long long N, int H, int W) {
    if (N <= 0 || H <= 0 || W <= 0 || N > 65535 || (long long)H * W >= (1ll << 30)) {
        set_error("bad tile geometry (need 1 <= N <= 65535, H*W < 2^30)");
        return TISEG_ERR_ARG;
    }
    return TISEG_OK;
}

// ---- one call of a C entry point --------------------------------------------------------------------------------
//   Call call(c, "tiseg_x", N, H, W);        checks the context and the geometry, then resets the arena
//   d_a = call.in(a, n); d_b = call.out(b, n);   device pointers pass through, host arguments are staged
//   TISEG_TRY(call.status());                once, after the staging and before the first launch
//   return call.finish();                    the copies back to host outputs, and the wait for them
// in / out / inout return nullptr for a null argument and only then, so an optional argument cannot be mistaken for
// a failed staging.  The first failure (bad geometry, workspace allocation, host-to-device copy) is recorded with its
// message; nothing is staged after it, and every later argument comes back as given, which no launch may use before
// status() is checked.  There is no destructor: a call that returns early leaves its pending copies to the next call,
// which drops them.
class Call {
  public:
    // `variants`: images per tile (test-time augmentation); the geometry check counts N * variants tiles
    Call(tiseg_ctx* c, const char* name, int N, int H, int W, int variants = 1);
    Geom g{};                   // of the N tiles (all zero if the geometry was refused)
    size_t total = 0;           // N * H * W
    template <class T> const T* in(const T* p, size_t n) { return (const T*)stage(const_cast<T*>(p), n * sizeof(T), true, false); }
    const void* in_bytes(const void* p, size_t bytes) { return stage(const_cast<void*>(p), bytes, true, false); }
    template <class T> T* out(T* p, size_t n) { return (T*)stage(p, n * sizeof(T), false, true); }
    template <class T> T* inout(T* p, size_t n) { return (T*)stage(p, n * sizeof(T), true, true); }
    int status() const;         // the recorded failure (its message becomes the last error), or TISEG_OK
    int finish();               // status(), or: queue the copies back to host outputs and wait for them

  private:
    tiseg_ctx* c_;
    int err_ = TISEG_OK;
    std::string msg_;
    void* stage(void* p, size_t bytes, bool to_device, bool to_host);
    void* failed(void* p, int err);
};

#ifdef __CUDACC__
struct Pix {
    int n, y, x;               // tile, row, column (x may be >= W on the ragged last segment)
    long long base;            // n * P
    int idx;                   // y * W + x  (tile-local flat index)
    int lane;
    bool ok;                   // x < W
};
// returns false if this warp has no work (uniform across the warp)
__device__ __forceinline__ bool warp_pixel(const Geom& g, Pix& p) {
    int w = blockIdx.x * TISEG_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    p.lane = threadIdx.x & 31;
    if (w >= g.wpt) return false;
    p.n = blockIdx.y;
    p.y = w / g.SEG;
    p.x = (w - p.y * g.SEG) * 32 + p.lane;
    p.ok = p.x < g.W;
    p.base = (long long)p.n * g.P;
    p.idx = p.y * g.W + p.x;
    return true;
}

// ---- strip iteration: one warp = STRIP_R consecutive rows of one 32-column segment -----------------------
// Loads of the STRIP_R rows are issued before any of them is consumed (independent requests in flight), and
// 3x3 stencils reuse the rows they share.  Consecutive warps take consecutive segments of the same row chunk.
#define STRIP_R 4
struct Strip {
    int n, x, y0, seg, lane;   // tile, column of this lane, first row, segment index
    bool okx;                  // x < W
    long long base;            // n * P
};
inline dim3 strip_grid(const Geom& g) {
    long long warps = (long long)g.SEG * ((g.H + STRIP_R - 1) / STRIP_R);
    return dim3((unsigned)((warps + TISEG_WARPS_PER_BLOCK - 1) / TISEG_WARPS_PER_BLOCK), grid_tiles(g), 1);
}
#ifdef __CUDACC__
// tile handled in iteration t of a FOR_TILES loop: the block's own tile (once), or entry t of the tile list.
// LISTED is a compile-time flag of the kernel, so the ordinary instantiation keeps its single straight-line pass
__device__ __forceinline__ int tile_listed(const Geom& g, int t) { return t < *g.tn ? g.tl[t] : -1; }
#define FOR_TILES_OF(LISTED, g, own, n) \
    for (int _t = 0, n = (LISTED) ? ::tiseg::tile_listed(g, 0) : (own); n >= 0; n = (LISTED) ? ::tiseg::tile_listed(g, ++_t) : -1)
#define FOR_TILES(LISTED, g, n) FOR_TILES_OF(LISTED, g, (int)blockIdx.y, n)
// launch kern<false> on every tile, or kern<true> on the tile list of g
#define TISEG_LAUNCH_TILES(c, kern, g, grid, block, smem, ...)                                          \
    do {                                                                                                \
        if ((g).tl) TISEG_LAUNCH(c, kern<true>, grid, block, smem, __VA_ARGS__);                        \
        else TISEG_LAUNCH(c, kern<false>, grid, block, smem, __VA_ARGS__);                              \
    } while (0)
__device__ __forceinline__ void strip_set_tile(const Geom& g, Strip& s, int n) { s.n = n; s.base = (long long)n * g.P; }
__device__ __forceinline__ bool warp_strip(const Geom& g, Strip& s) {
    int w = blockIdx.x * TISEG_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    s.lane = threadIdx.x & 31;
    int chunks = (g.H + STRIP_R - 1) / STRIP_R;
    if (w >= g.SEG * chunks) return false;
    int ch = w / g.SEG;
    s.seg = w - ch * g.SEG;
    s.y0 = ch * STRIP_R;
    s.n = blockIdx.y;
    s.x = s.seg * 32 + s.lane;
    s.okx = s.x < g.W;
    s.base = (long long)s.n * g.P;
    return true;
}
// centre / left / right columns of rows y0-1 .. y0+STRIP_R for a 3x3 stencil; out-of-image taps read `oob`.
// Split in two so a kernel can look at the centre rows first and skip the halo work of an empty strip.
template <class T>
__device__ __forceinline__ void strip_load_c(const Geom& g, const Strip& s, const T* __restrict__ tile, T oob,
                                             T (&c)[STRIP_R + 2]) {
#pragma unroll
    for (int j = 0; j < STRIP_R + 2; ++j) {
        int y = s.y0 - 1 + j;
        c[j] = (y >= 0 && y < g.H && s.okx) ? tile[y * g.W + s.x] : oob;
    }
}
template <class T>
__device__ __forceinline__ void strip_fill_lr(const Geom& g, const Strip& s, const T* __restrict__ tile, T oob,
                                              const T (&c)[STRIP_R + 2], T (&l)[STRIP_R + 2], T (&r)[STRIP_R + 2]) {
#pragma unroll
    for (int j = 0; j < STRIP_R + 2; ++j) {
        int y = s.y0 - 1 + j;
        bool oky = y >= 0 && y < g.H;
        T el = oob, er = oob;
        if (s.lane == 0 && oky && s.x > 0 && s.x - 1 < g.W) el = tile[y * g.W + s.x - 1];
        if (s.lane == 31 && oky && s.x + 1 < g.W) er = tile[y * g.W + s.x + 1];
        l[j] = el; r[j] = er;
    }
#pragma unroll
    for (int j = 0; j < STRIP_R + 2; ++j) {
        T a = __shfl_up_sync(0xffffffffu, c[j], 1), b = __shfl_down_sync(0xffffffffu, c[j], 1);
        if (s.lane != 0) l[j] = a;
        if (s.lane != 31) r[j] = b;
    }
}
template <class T>
__device__ __forceinline__ void strip_load3(const Geom& g, const Strip& s, const T* __restrict__ tile, T oob,
                                            T (&c)[STRIP_R + 2], T (&l)[STRIP_R + 2], T (&r)[STRIP_R + 2]) {
    strip_load_c<T>(g, s, tile, oob, c);
    strip_fill_lr<T>(g, s, tile, oob, c, l, r);
}
#endif

// ---- flat elementwise iteration: one thread = 4 consecutive elements (128-bit fp32/int32, 32-bit uint8) ----
// `vec` (uniform) says every pointer of the launch is 16-byte aligned; otherwise, and on the ragged tail, the
// accessors fall back to scalar loads.  Four elements per thread keeps 16 B per request in flight, which is what
// a pure streaming pass needs to approach HBM bandwidth (one 4-byte load per thread cannot cover the latency).
template <class T> struct Pack4 { T v[4]; };
template <> struct __align__(16) Pack4<float> { float v[4]; };
template <> struct __align__(16) Pack4<int> { int v[4]; };
template <> struct __align__(4) Pack4<uint8_t> { uint8_t v[4]; };

template <class T>
__device__ __forceinline__ Pack4<T> ld4(const T* __restrict__ p, long long i, long long total, bool vec) {
    Pack4<T> r;
    if (vec && i + 3 < total) r = *reinterpret_cast<const Pack4<T>*>(p + i);
    else {
#pragma unroll
        for (int k = 0; k < 4; ++k) r.v[k] = i + k < total ? p[i + k] : T(0);
    }
    return r;
}
template <class T>
__device__ __forceinline__ void st4(T* __restrict__ p, long long i, long long total, bool vec, const Pack4<T>& r) {
    if (vec && i + 3 < total) *reinterpret_cast<Pack4<T>*>(p + i) = r;
    else {
#pragma unroll
        for (int k = 0; k < 4; ++k) if (i + k < total) p[i + k] = r.v[k];
    }
}
__device__ __forceinline__ long long flat4_index() { return ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4; }

// ---- network outputs in fp32, fp16 or bf16 (TISEG_DTYPE_*) ---------------------------------------------------------
// Kernels that read a network output are templated on its element type and convert at the load; everything after the
// load is fp32 arithmetic.  fp16 -> fp32 and bf16 -> fp32 are exact, so a half input gives the bits of its fp32 upcast.
template <> struct __align__(8) Pack4<__half> { __half v[4]; };
template <> struct __align__(8) Pack4<__nv_bfloat16> { __nv_bfloat16 v[4]; };
template <class T> struct InType;
template <> struct InType<float> { static constexpr int code = TISEG_DTYPE_F32; };
template <> struct InType<__half> { static constexpr int code = TISEG_DTYPE_F16; };
template <> struct InType<__nv_bfloat16> { static constexpr int code = TISEG_DTYPE_BF16; };
// timing name of a launch: the fp32 instantiation keeps the plain kernel name, the half ones carry the dtype
#define TISEG_IN_NAME(T, name) \
    (::tiseg::InType<T>::code == TISEG_DTYPE_F32 ? name : ::tiseg::InType<T>::code == TISEG_DTYPE_F16 ? name ":f16" : name ":bf16")
// four consecutive elements of a network output are 16 B in fp32, 8 B in half precision
template <class T> inline bool aligned_x4(const void* p) { return (((uintptr_t)p) & (4 * sizeof(T) - 1)) == 0; }
inline int check_dtype(int dtype, const char* where) {
    if (dtype == TISEG_DTYPE_F32 || dtype == TISEG_DTYPE_F16 || dtype == TISEG_DTYPE_BF16) return TISEG_OK;
    set_error(std::string(where) + ": unknown dtype code " + std::to_string(dtype) + " (0 fp32, 1 fp16, 2 bf16)");
    return TISEG_ERR_ARG;
}
inline size_t dtype_bytes(int dtype) { return dtype == TISEG_DTYPE_F32 ? 4 : 2; }
// call fn(T()) with T the element type of the dtype code (checked beforehand with check_dtype)
template <class F> inline int with_dtype(int dtype, F&& fn) {
    if (dtype == TISEG_DTYPE_F16) return fn(__half());
    if (dtype == TISEG_DTYPE_BF16) return fn(__nv_bfloat16());
    return fn(0.f);
}

__device__ __forceinline__ float to_f32(float x) { return x; }
__device__ __forceinline__ float to_f32(__half x) { return __half2float(x); }
__device__ __forceinline__ float to_f32(__nv_bfloat16 x) { return __bfloat162float(x); }
__device__ __forceinline__ float2 to_f32(float2 x) { return x; }
__device__ __forceinline__ float2 to_f32(__half2 x) { return __half22float2(x); }
__device__ __forceinline__ float2 to_f32(__nv_bfloat162 x) { return __bfloat1622float2(x); }
template <class T> struct Pair;                        // two interleaved channels (an HWC map of two)
template <> struct Pair<float> { typedef float2 type; };
template <> struct Pair<__half> { typedef __half2 type; };
template <> struct Pair<__nv_bfloat16> { typedef __nv_bfloat162 type; };

// ld4 of a network output, converted to fp32 (`vec`: the pointer is aligned to four elements)
__device__ __forceinline__ Pack4<float> ld4f(const float* __restrict__ p, long long i, long long total, bool vec) {
    return ld4(p, i, total, vec);
}
template <class T>
__device__ __forceinline__ Pack4<float> ld4f(const T* __restrict__ p, long long i, long long total, bool vec) {
    Pack4<float> r;
    if (vec && i + 3 < total) {
        const Pack4<T> h = *reinterpret_cast<const Pack4<T>*>(p + i);
#pragma unroll
        for (int k = 0; k < 4; ++k) r.v[k] = to_f32(h.v[k]);
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) r.v[k] = i + k < total ? to_f32(p[i + k]) : 0.f;
    }
    return r;
}
// four aligned consecutive elements, converted to fp32
__device__ __forceinline__ void ld4f_aligned(const float* p, float (&x)[4]) {
    const float4 u = *reinterpret_cast<const float4*>(p);
    x[0] = u.x; x[1] = u.y; x[2] = u.z; x[3] = u.w;
}
template <class T>
__device__ __forceinline__ void ld4f_aligned(const T* p, float (&x)[4]) {
    const Pack4<T> h = *reinterpret_cast<const Pack4<T>*>(p);
#pragma unroll
    for (int k = 0; k < 4; ++k) x[k] = to_f32(h.v[k]);
}

// ---- instance maps in int32 or uint16 -----------------------------------------------------------------------------------
// Kernels that read a ground-truth instance map are templated on its id type: int32, or uint16 (ids below 65536, which
// every dataset the reference converts keeps to) read as it is, at half the bytes, and widened in registers.  A uint16 id
// is below every id table's VM = max(H*W + 1, 65536), so it can never raise the "instance id out of range" error.
// Timing name of a launch: the int32 instantiation keeps the plain kernel name, the uint16 one carries the type.
#define TISEG_ID_NAME(T, name) (sizeof(T) == 2 ? name "<uint16_t>" : name)
// four consecutive ids from an address aligned to four elements: one 16-byte load in int32, one 8-byte load in uint16
__device__ __forceinline__ void ld_ids4(const int32_t* p, int (&v)[4]) {
    const int4 q = *reinterpret_cast<const int4*>(p);
    v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
}
__device__ __forceinline__ void ld_ids4(const uint16_t* p, int (&v)[4]) {
    const uint2 q = *reinterpret_cast<const uint2*>(p);
    v[0] = q.x & 0xffffu; v[1] = q.x >> 16; v[2] = q.y & 0xffffu; v[3] = q.y >> 16;
}

// Given the ballot of "this lane continues the run of the lane to its left" (bit 0 of the segment may be
// set when the run continues from the previous segment), the lane at which my run starts inside the segment.
__device__ __forceinline__ int run_start_lane(unsigned cont, int lane) {
    unsigned brk = ~cont & (0xffffffffu >> (31 - lane));   // lanes <= me that start a run
    return brk ? 31 - __clz(brk) : 0;
}
// number of lanes in my run from its start (inside the segment) to its end, valid at any lane of the run
__device__ __forceinline__ int run_end_lane(unsigned cont, int lane) {
    unsigned brk = ~cont & ~(0xffffffffu >> (31 - lane));  // lanes > me that start a run
    return brk ? (__ffs(brk) - 1) - 1 : 31;
}

// ---- rows as quads: one warp = 128 pixels of a row, four per thread -------------------------------------------
// The pixel-per-lane kernels of this library were issue-bound (ncu: 70-85 % issue slots at a quarter of the HBM
// rate); the per-run kernels therefore read four pixels per thread and still post ONE set of atomics per run of
// equal keys inside the warp's 128 pixels.
struct Quad { int n, y, x, lane; long long base; };      // x = the first of the thread's four columns
inline dim3 quad_grid(const Geom& g) {
    long long warps = (long long)((g.W + 127) / 128) * g.H;
    return dim3((unsigned)((warps + TISEG_WARPS_PER_BLOCK - 1) / TISEG_WARPS_PER_BLOCK), grid_tiles(g), 1);
}
__device__ __forceinline__ bool warp_quad(const Geom& g, Quad& q) {
    const int segs = (g.W + 127) >> 7;
    const long long w = (long long)blockIdx.x * TISEG_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    if (w >= (long long)segs * g.H) return false;
    q.lane = threadIdx.x & 31;
    q.n = blockIdx.y;
    q.y = (int)(w / segs);
    q.x = (int)(w - (long long)q.y * segs) * 128 + q.lane * 4;
    q.base = (long long)q.n * g.P;
    return true;
}
__device__ __forceinline__ void quad_load_i32(const Geom& g, const Quad& q, const int32_t* __restrict__ tile, int oob, bool vec, int (&v)[4]) {
    const int32_t* rp = tile + (long long)q.y * g.W + q.x;
    if (vec && q.x + 3 < g.W) { const int4 t = *reinterpret_cast<const int4*>(rp); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w; }
    else {
#pragma unroll
        for (int k = 0; k < 4; ++k) v[k] = q.x + k < g.W ? rp[k] : oob;
    }
}
// runs of equal keys along the warp's 128 pixels; `null` keys belong to no run
struct QuadRuns {
    unsigned fg, cont;      // bit k: pixel k has a key / continues the run of the pixel to its left
    int ext;                // pixels beyond my pixel 3 that belong to its run
};
template <class K>
__device__ __forceinline__ QuadRuns quad_runs(const K (&key)[4], K null, int lane) {
    QuadRuns r;
    const K left = __shfl_up_sync(0xffffffffu, key[3], 1);
    r.fg = (key[0] != null ? 1u : 0u) | (key[1] != null ? 2u : 0u) | (key[2] != null ? 4u : 0u) | (key[3] != null ? 8u : 0u);
    r.cont = (((lane > 0 && key[0] == left) ? 1u : 0u) | (key[1] == key[0] ? 2u : 0u) | (key[2] == key[1] ? 4u : 0u) |
              (key[3] == key[2] ? 8u : 0u)) & r.fg;
    const unsigned full = __ballot_sync(0xffffffffu, r.cont == 15u);
    const unsigned rest = lane < 31 ? full >> (lane + 1) : 0u;
    const int nfull = __ffs(~rest) - 1, next = lane + 1 + nfull;
    const int lead = __ffs(~r.cont) - 1;                                   // my leading continuing pixels
    const int nl = __shfl_sync(0xffffffffu, lead, next < 32 ? next : 31);
    r.ext = 4 * nfull + (next < 32 ? nl : 0);
    return r;
}
// iterate the runs that START in this thread: k = first pixel, len = length inside the warp's 128 pixels
#define FOR_QUAD_RUNS(r, k, len)                                                                             \
    for (unsigned _s = (r).fg & ~(r).cont, k = 0, len = 0;                                                   \
         _s && (k = __ffs(_s) - 1, len = __ffs(~((r).cont >> (k + 1))), len += (k + len == 4 ? (r).ext : 0), true); _s &= _s - 1)

// (no __restrict__/const: parents are updated concurrently, loads must stay coherent)
__device__ __forceinline__ int uf_find(int* par, int x) {
    int p = par[x];
    while (p != x) { x = p; p = par[x]; }
    return x;
}
// union by minimum index: the root of a component is its lowest flat index (= first pixel in raster order)
__device__ __forceinline__ void uf_union(int* par, int a, int b) {
    for (;;) {
        a = uf_find(par, a);
        b = uf_find(par, b);
        if (a == b) return;
        if (a < b) { int t = a; a = b; b = t; }      // a > b: hang a under b
        int old = atomicMin(&par[a], b);
        if (old == a) return;
        a = old;
    }
}
#endif

}  // namespace tiseg
