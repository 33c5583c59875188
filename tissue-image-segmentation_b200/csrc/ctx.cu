// Context, error reporting and the call-scoped device workspace of libtiseg_b200.so.
#include <cstdio>
#include <cstring>

#include "common.cuh"

namespace tiseg {

static thread_local std::string g_err;

void set_error(const std::string& msg) { g_err = msg; }

int fail(const char* where, cudaError_t e) {
    g_err = std::string(where) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")";
    return TISEG_ERR_CUDA;
}

void* ws_alloc(tiseg_ctx* c, size_t bytes) {
    bytes = (bytes + 255) & ~size_t(255);
    if (bytes == 0) bytes = 256;
    while (c->cur_block < c->blocks.size()) {
        auto& b = c->blocks[c->cur_block];
        if (c->cur_off + bytes <= b.cap) {
            void* r = b.p + c->cur_off;
            c->cur_off += bytes;
            return r;
        }
        c->cur_block++;
        c->cur_off = 0;
    }
    size_t cap = bytes > (size_t(256) << 20) ? bytes : (size_t(256) << 20);
    char* p = nullptr;
    if (cudaMalloc(&p, cap) != cudaSuccess) {
        cudaGetLastError();
        set_error("workspace cudaMalloc failed");
        return nullptr;
    }
    c->blocks.push_back({p, cap});
    c->cur_block = c->blocks.size() - 1;
    c->cur_off = bytes;
    return p;
}

static bool is_device_ptr(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

Call::Call(tiseg_ctx* c, const char* name, int N, int H, int W, int variants) : c_(c) {
    if (!c) {
        err_ = TISEG_ERR_ARG;
        msg_ = std::string(name) + ": null context";
        return;
    }
    if ((err_ = check_geom((long long)N * variants, H, W)) != TISEG_OK) {
        msg_ = g_err;
        return;
    }
    cudaSetDevice(c->device);
    // coalesce the arena if the previous call spilled into extra blocks
    if (c->blocks.size() > 1) {
        size_t total = 0;
        for (auto& b : c->blocks) total += b.cap;
        cudaStreamSynchronize(c->stream);
        for (auto& b : c->blocks) cudaFree(b.p);
        c->blocks.clear();
        char* p = nullptr;
        if (cudaMalloc(&p, total) == cudaSuccess) c->blocks.push_back({p, total});
        else cudaGetLastError();
    }
    c->cur_block = 0;
    c->cur_off = 0;
    c->pending.clear();
    g = make_geom(N, H, W);
    total = (size_t)N * g.P;
}

void* Call::failed(void* p, int err) {
    err_ = err;
    msg_ = g_err;
    return p;
}

// device pointers are returned as they are; a host argument gets arena scratch, filled with an async H2D if it is
// read (to_device) and copied back by finish() if it is written (to_host)
void* Call::stage(void* p, size_t bytes, bool to_device, bool to_host) {
    if (!p || err_ != TISEG_OK || is_device_ptr(p)) return p;
    void* d = ws_alloc(c_, bytes);
    if (!d) return failed(p, TISEG_ERR_CUDA);
    if (to_device && cudaMemcpyAsync(d, p, bytes, cudaMemcpyHostToDevice, c_->stream) != cudaSuccess)
        return failed(p, fail("H2D", cudaGetLastError()));
    if (to_host) c_->pending.push_back({p, d, bytes});
    return d;
}

int Call::status() const {
    if (err_ != TISEG_OK) set_error(msg_);
    return err_;
}

int Call::finish() {
    if (err_ != TISEG_OK) return status();
    tiseg_ctx* c = c_;
    if (c->pending.empty()) return TISEG_OK;          // device outputs: stream-ordered, nothing to wait for
    for (auto& q : c->pending)
        TISEG_CHECK(cudaMemcpyAsync(q.host, q.dev, q.bytes, cudaMemcpyDeviceToHost, c->stream));
    c->pending.clear();
    TISEG_CHECK(cudaMemcpyAsync(c->h_err, c->d_err, 2 * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    TISEG_CHECK(cudaStreamSynchronize(c->stream));
    return check_deferred(c);
}

int check_deferred(tiseg_ctx* c) {
    if (!c->h_err[0] && !c->h_err[1]) return TISEG_OK;
    const bool range = c->h_err[0] != 0;
    c->h_err[0] = c->h_err[1] = 0;
    cudaMemsetAsync(c->d_err, 0, 2 * sizeof(int), c->stream);
    set_error(range ? "instance id out of the supported range (need 0 <= id < max(H*W+1, 65536))"
                    : "internal pair table lost an entry");
    return TISEG_ERR_LIMIT;
}

int zero(tiseg_ctx* c, void* p, size_t bytes) {
    cudaEvent_t tb = c->timing ? timing_before(c, "memset") : nullptr;
    TISEG_CHECK(cudaMemsetAsync(p, 0, bytes, c->stream));
    if (tb) cudaEventRecord(tb, c->stream);
    return TISEG_OK;
}

static cudaEvent_t get_event(tiseg_ctx* c) {
    if (!c->event_pool.empty()) { cudaEvent_t e = c->event_pool.back(); c->event_pool.pop_back(); return e; }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}

cudaEvent_t timing_before(tiseg_ctx* c, const char* name) {
    tiseg_ctx::Timed t;
    t.name = name; t.a = get_event(c); t.b = get_event(c);
    cudaEventRecord(t.a, c->stream);
    c->timed.push_back(t);
    return t.b;
}

}  // namespace tiseg

extern "C" {

int tiseg_create(tiseg_ctx** out, int device) {
    if (!out) { tiseg::set_error("tiseg_create: null out"); return TISEG_ERR_ARG; }
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
        cudaGetLastError();
        tiseg::set_error("tiseg_create: no CUDA device (libtiseg_b200 has no CPU fallback)");
        return TISEG_ERR_NOGPU;
    }
    if (device < 0 || device >= n) { tiseg::set_error("tiseg_create: bad device index"); return TISEG_ERR_ARG; }
    TISEG_CHECK(cudaSetDevice(device));
    tiseg_ctx* c = new tiseg_ctx();
    c->device = device;
    cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { delete c; return tiseg::fail("cudaStreamCreate", e); }
    c->own_stream = true;
    cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (cudaMalloc(&c->d_err, 2 * sizeof(int)) != cudaSuccess || cudaMemset(c->d_err, 0, 2 * sizeof(int)) != cudaSuccess ||
        cudaHostAlloc(&c->h_err, 2 * sizeof(int), cudaHostAllocDefault) != cudaSuccess) {
        cudaError_t e2 = cudaGetLastError();
        tiseg_destroy(c);
        return tiseg::fail("tiseg_create", e2);
    }
    c->h_err[0] = c->h_err[1] = 0;
    *out = c;
    return TISEG_OK;
}

int tiseg_destroy(tiseg_ctx* c) {
    if (!c) return TISEG_OK;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    for (auto& b : c->blocks) cudaFree(b.p);
    if (c->d_err) cudaFree(c->d_err);
    if (c->h_err) cudaFreeHost(c->h_err);
    if (c->order_ev) cudaEventDestroy(c->order_ev);
    if (c->own_stream) cudaStreamDestroy(c->stream);
    delete c;
    return TISEG_OK;
}

int tiseg_set_stream(tiseg_ctx* c, void* s) {
    if (!c) { tiseg::set_error("null ctx"); return TISEG_ERR_ARG; }
    cudaSetDevice(c->device);
    cudaStream_t ns = (cudaStream_t)s;   // NULL == the legacy default stream (what torch uses by default)
    if (c->own_stream) {
        cudaStreamSynchronize(c->stream);
        cudaStreamDestroy(c->stream);
        c->own_stream = false;
    } else if (ns != c->stream) {
        // Work queued on the previous stream may still be using the arena that the next call on the new stream resets
        // and overwrites: order the new stream after it (event, no host wait).  A stream under graph capture cannot
        // wait on an event from outside the capture; callers that capture keep one context per stream (_lib.lane).
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(ns, &cs) != cudaSuccess) { cudaGetLastError(); cs = cudaStreamCaptureStatusNone; }
        if (cs == cudaStreamCaptureStatusNone) {
            if (!c->order_ev && cudaEventCreateWithFlags(&c->order_ev, cudaEventDisableTiming) != cudaSuccess) {
                cudaGetLastError();
                c->order_ev = nullptr;
            }
            if (c->order_ev) {
                if (cudaEventRecord(c->order_ev, c->stream) == cudaSuccess) cudaStreamWaitEvent(ns, c->order_ev, 0);
                else { cudaGetLastError(); cudaStreamSynchronize(c->stream); cudaGetLastError(); }
            }
        }
    }
    c->stream = ns;
    return TISEG_OK;
}

int tiseg_synchronize(tiseg_ctx* c) {
    if (!c) { tiseg::set_error("null ctx"); return TISEG_ERR_ARG; }
    TISEG_CHECK(cudaMemcpyAsync(c->h_err, c->d_err, 2 * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    TISEG_CHECK(cudaStreamSynchronize(c->stream));
    return tiseg::check_deferred(c);
}

int tiseg_timing_enable(tiseg_ctx* c, int on) {
    if (!c) { tiseg::set_error("null ctx"); return TISEG_ERR_ARG; }
    c->timing = on != 0;
    return TISEG_OK;
}

// "name count total_ms\n" per kernel, aggregated over everything launched since timing was enabled
int tiseg_timing_report(tiseg_ctx* c, char* buf, int cap) {
    if (!c || !buf || cap <= 0) { tiseg::set_error("tiseg_timing_report: bad argument"); return TISEG_ERR_ARG; }
    TISEG_CHECK(cudaStreamSynchronize(c->stream));
    struct Agg { const char* name; long long n; double ms; };
    std::vector<Agg> agg;
    for (auto& t : c->timed) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, t.a, t.b);
        size_t i = 0;
        for (; i < agg.size(); ++i) if (!strcmp(agg[i].name, t.name)) break;
        if (i == agg.size()) agg.push_back({t.name, 0, 0.0});
        agg[i].n++; agg[i].ms += ms;
        c->event_pool.push_back(t.a); c->event_pool.push_back(t.b);
    }
    c->timed.clear();
    std::string out;
    char line[256];
    for (auto& a : agg) { snprintf(line, sizeof line, "%s %lld %.6f\n", a.name, a.n, a.ms); out += line; }
    if ((int)out.size() + 1 > cap) { tiseg::set_error("tiseg_timing_report: buffer too small"); return TISEG_ERR_ARG; }
    memcpy(buf, out.c_str(), out.size() + 1);
    return TISEG_OK;
}

const char* tiseg_last_error(void) { return tiseg::g_err.c_str(); }

long long tiseg_launch_count(tiseg_ctx* c) { return c ? c->launches : 0; }

int tiseg_version(void) { return 300; }

#ifndef TISEG_SRC_HASH
#define TISEG_SRC_HASH "unknown"
#endif
const char* tiseg_build_hash(void) { return TISEG_SRC_HASH; }

}  // extern "C"
