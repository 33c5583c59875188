// K10 — align_foreground (tiseg/models/utils/postprocess.py:123-155) and the multi-task postprocess built on it
// (multi_task_unet.py:84-106, multi_task_cunet.py:86-108, multi_task_cdnet.py:222-243).
//
// align_foreground is an ORDERED multi-source BFS: the queue starts with every labelled pixel in raster order;
// in each of at most time-1 rounds every queued pixel, in queue order, claims its still-unlabelled foreground
// 8-neighbours (direction order k = 1..8) and appends them.  A pixel takes the label of the FIRST claimant,
// so the result depends on the queue order.  The order restricted to one 8-connected component of
// (labelled | foreground) does not depend on the other components, so each component ("blob") is flooded
// sequentially by one warp with its own FIFO slice — the same decomposition as the watershed (watershed.cuh).
#include "ccl.cuh"
#include "morph.cuh"
#include "watershed.cuh"

namespace tiseg {

#define FULL 0xffffffffu

__global__ void __launch_bounds__(TISEG_THREADS)
k_align_bfs(Geom g, const uint8_t* __restrict__ fgm, const int* __restrict__ par, BlobInfo b, int* work, int* queue,
            int32_t* pred, int time) {
    const int lane = threadIdx.x & 31;
    const int n = blockIdx.y;
    const int B = b.count[n];
    const long long base = (long long)n * g.P, ko = (long long)n * b.KS;
    const uint8_t* fg = fgm + base;
    const int* tp = par + base;
    int32_t* o = pred + base;
    const int W = g.W, H = g.H;
    // (row, col) offsets for k = 1..8: postprocess.py:128-129
    const int dr[8] = {0, -1, -1, -1, 0, 1, 1, 1};
    const int dc[8] = {-1, -1, 0, 1, 1, 1, 0, -1};
    for (;;) {
        int bid = 0;
        if (lane == 0) bid = atomicAdd(&work[n], 1) + 1;
        bid = __shfl_sync(FULL, bid, 0);
        if (bid > B) break;
        const int root = b.root[ko + bid];
        const int y0 = root / W, y1 = b.ymax[ko + bid], x0 = b.xmin[ko + bid], x1 = b.xmax[ko + bid];
        int* q = queue + base + b.off[ko + bid];
        int tail = 0;
        for (int y = y0; y <= y1; ++y) {
            for (int xb = x0; xb <= x1; xb += 32) {
                int x = xb + lane;
                bool seed = false;
                if (x <= x1) { int idx = y * W + x; seed = tp[idx] == root && o[idx] > 0; }
                unsigned m = __ballot_sync(FULL, seed);
                if (seed) q[tail + __popc(m & ((1u << lane) - 1))] = y * W + x;
                tail += __popc(m);
            }
        }
        __syncwarp();
        if (lane == 0) {
            int start = 0, end = tail, iter = 1;
            while (end > start) {
                if (iter >= time) break;
                ++iter;
                for (int ix = start; ix < end; ++ix) {
                    const int pix = q[ix];
                    const int lab = o[pix];
                    const int r = pix / W, cc = pix - r * W;
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        int nr = r + dr[k], nc = cc + dc[k];
                        if (nr < 0 || nr >= H || nc < 0 || nc >= W) continue;
                        int nb = nr * W + nc;
                        if (o[nb] == 0 && fg[nb] > 0) { q[tail++] = nb; o[nb] = lab; }
                    }
                }
                start = end;
                end = tail;
            }
        }
        __syncwarp();
    }
}

int align_foreground_dev(tiseg_ctx* c, const Geom& g, int32_t* pred, const uint8_t* fg, int time) {
    size_t total = (size_t)g.N * g.P;
    int* par = ws<int>(c, total);
    int* rank = ws<int>(c, total);
    int* queue = ws<int>(c, total);
    int* work = ws<int>(c, (size_t)g.N);
    if (!par || !rank || !queue || !work) return TISEG_ERR_CUDA;
    BlobInfo b;
    TISEG_TRY(blobs_build(c, g, ImgOrI32U8{pred, fg}, par, rank, b, true, 2));
    TISEG_TRY(zero(c, work, (size_t)g.N * sizeof(int)));
    int per_tile = (c->sm_count * 8 * 4 + g.N - 1) / g.N;
    per_tile = per_tile < 1 ? 1 : (per_tile > 512 ? 512 : per_tile);
    TISEG_LAUNCH(c, k_align_bfs, dim3(per_tile, g.N), TISEG_THREADS, 0, g, fg, par, b, work, queue, pred, time);
    return TISEG_OK;
}

__global__ void k_class_mask(Geom g, const uint8_t* __restrict__ cls, int id, uint8_t* __restrict__ out) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    out[px.base + px.idx] = cls[px.base + px.idx] == id;
}
__global__ void k_paint_class(Geom g, const uint8_t* __restrict__ m, int id, uint8_t* canvas) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    if (m[px.base + px.idx]) canvas[px.base + px.idx] = (uint8_t)id;
}

// sem canvas: per class ascending, remove_small_objects(5) THEN binary_fill_holes, later classes overwrite
int sem_canvas_dev(tiseg_ctx* c, const Geom& g, const uint8_t* sem, int max_class, uint8_t* canvas) {
    size_t total = (size_t)g.N * g.P;
    uint8_t* m0 = ws<uint8_t>(c, total);
    uint8_t* m1 = ws<uint8_t>(c, total);
    uint8_t* m2 = ws<uint8_t>(c, total);
    int* par = ws<int>(c, total);
    if (!m0 || !m1 || !m2 || !par) return TISEG_ERR_CUDA;
    TISEG_TRY(zero(c, canvas, total));
    for (int id = 1; id <= max_class; ++id) {
        TISEG_LAUNCH(c, k_class_mask, warp_grid(g), TISEG_THREADS, 0, g, sem, id, m0);
        TISEG_TRY(remove_small_mask(c, g, m0, 5, 1, m1));
        TISEG_TRY(ccl_build(c, g, ImgNotMaskU8{m1}, 1, par));
        TISEG_TRY(fill_from_complement_forest(c, g, par, m2));
        TISEG_LAUNCH(c, k_paint_class, warp_grid(g), TISEG_THREADS, 0, g, m2, id, canvas);
    }
    return TISEG_OK;
}

}  // namespace tiseg

using namespace tiseg;

extern "C" {

int tiseg_align_foreground(tiseg_ctx* c, int32_t* pred, const uint8_t* foreground, int N, int H, int W, int time) {
    if (!c || !pred || !foreground) { set_error("tiseg_align_foreground: bad argument"); return TISEG_ERR_ARG; }
    Call call(c, "tiseg_align_foreground", N, H, W);
    int32_t* d_pred = call.inout(pred, call.total);
    const uint8_t* d_fg = call.in(foreground, call.total);
    TISEG_TRY(call.status());
    TISEG_TRY(align_foreground_dev(c, call.g, d_pred, d_fg, time));
    return call.finish();
}

int tiseg_postproc_multitask(tiseg_ctx* c, const uint8_t* inner, const uint8_t* sem, int N, int H, int W,
                             int max_class, int edge_id, int time, uint8_t* canvas_out, int32_t* inst_out) {
    if (!c || !inner || !sem || !canvas_out || !inst_out || max_class < 1 || max_class > 63) {
        set_error("tiseg_postproc_multitask: bad argument");
        return TISEG_ERR_ARG;
    }
    Call call(c, "tiseg_postproc_multitask", N, H, W);
    const uint8_t* d_inner = call.in(inner, call.total);
    const uint8_t* d_sem = call.in(sem, call.total);
    uint8_t* d_canvas = call.out(canvas_out, call.total);
    int32_t* d_inst = call.out(inst_out, call.total);
    TISEG_TRY(call.status());
    const Geom& g = call.g;
    TISEG_TRY(sem_canvas_dev(c, g, d_sem, max_class, d_canvas));
    // measure.label(bin_pred, connectivity=1) with the edge class zeroed (multi_task_cunet.py:99-103)
    TISEG_TRY(ccl_label(c, g, ImgEqU8Drop{d_inner, edge_id}, 1, d_inst, nullptr));
    TISEG_TRY(align_foreground_dev(c, g, d_inst, d_canvas, time));
    return call.finish();
}

}  // extern "C"
