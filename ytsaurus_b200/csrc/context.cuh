// context.cuh — per-device context: stream, stream-ordered scratch memory, launch accounting, timers.
#pragma once

#include <mutex>
#include <vector>

#include "common.cuh"

namespace ytgpu {

struct TimedSpan {
    int cls;
    cudaEvent_t start, stop;
};

struct Context {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool owns_stream = false;
    u64 launches = 0;
    bool timers_enabled = false;
    std::vector<TimedSpan> spans;
    std::vector<float> pass_ms;  // one entry per radix pass launch (active and skipped)
    double ms[KC_COUNT] = {0};
    u64 timed_launches[KC_COUNT] = {0};
    u32* dev_err = nullptr;   // device error flag word
    u32* host_err = nullptr;  // pinned mirror
    // Entry points of the C ABI lock the context: the reference calls its readers / partitioners from several
    // threads (writer thread + SortInvoker pool), while the error words, timers and stream are per-context state.
    std::mutex mu;
    // cudaFuncSetAttribute applies to the CURRENT device only: every context raises the dynamic shared-memory
    // limits of the kernels it launches once (bit per kernel family), so a process may own contexts on several GPUs.
    u32 func_attrs_done = 0;
    int opt_merge_path = 1;    // ytgpu_merge_sorted_runs: 1 = merge-path rounds when the runs are few, 0 = always the stable sort
    bool last_merge_used_merge_path = false;
    int opt_sort_hybrid = 1;   // radix sort: 1 = hybrid MSD-prefix schedule when it applies, 0 = always full LSD

    Status alloc(void** p, size_t bytes) {
        if (bytes == 0) bytes = 16;
        cudaError_t e = cudaMallocAsync(p, bytes, stream);
        if (e == cudaErrorMemoryAllocation) {
            cudaGetLastError();
            return make_status(YTGPU_ERR_OUT_OF_MEMORY, "cudaMallocAsync(%zu bytes) failed", bytes);
        }
        if (e != cudaSuccess) return cuda_status(e, "cudaMallocAsync");
        return Status{};
    }
    void free(void* p) {
        if (p) cudaFreeAsync(p, stream);
    }
    void count_launch(int n = 1) { launches += (u64)n; }
    void collect_timers();
};

// RAII stream-ordered device buffer.
template <class T>
struct DevBuf {
    Context* ctx = nullptr;
    T* p = nullptr;
    size_t n = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf& operator=(DevBuf&& o) noexcept {
        if (this != &o) {
            reset();
            ctx = o.ctx;
            p = o.p;
            n = o.n;
            o.p = nullptr;
            o.n = 0;
        }
        return *this;
    }
    ~DevBuf() { reset(); }
    void reset() {
        if (p && ctx) ctx->free(p);
        p = nullptr;
        n = 0;
    }
    Status allocate(Context* c, size_t count) {
        reset();
        ctx = c;
        n = count;
        return c->alloc(reinterpret_cast<void**>(&p), count * sizeof(T));
    }
};

// Scoped CUDA-event span around one or more launches of a kernel class.
struct KernelTimer {
    Context* ctx;
    TimedSpan span;
    bool active;
    KernelTimer(Context* c, int cls, int launches = 1) : ctx(c), active(c->timers_enabled) {
        c->count_launch(launches);
        if (active) {
            span.cls = cls;
            cudaEventCreate(&span.start);
            cudaEventCreate(&span.stop);
            cudaEventRecord(span.start, c->stream);
            c->timed_launches[cls] += (u64)launches;
        }
    }
    ~KernelTimer() {
        if (active) {
            cudaEventRecord(span.stop, ctx->stream);
            ctx->spans.push_back(span);
        }
    }
};

// Move `bytes` between a caller buffer in `mem` space and device memory, on the context stream.
inline Status copy_in(Context* ctx, void* dst_dev, const void* src, size_t bytes, int mem) {
    if (bytes == 0) return Status{};
    YTGPU_CUDA_TRY(cudaMemcpyAsync(dst_dev, src, bytes,
                                   mem == YTGPU_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice,
                                   ctx->stream));
    return Status{};
}
inline Status copy_out(Context* ctx, void* dst, const void* src_dev, size_t bytes, int mem) {
    if (bytes == 0) return Status{};
    YTGPU_CUDA_TRY(cudaMemcpyAsync(dst, src_dev, bytes,
                                   mem == YTGPU_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice,
                                   ctx->stream));
    return Status{};
}

inline int fill_error(ytgpu_error* err, const Status& s) {
    if (err) {
        err->code = s.code;
        err->cuda_error = s.cuda;
        for (size_t i = 0; i < sizeof(err->message); ++i) err->message[i] = 0;
        for (size_t i = 0; i + 1 < sizeof(err->message) && s.msg[i]; ++i) err->message[i] = s.msg[i];
    }
    return s.code;
}

inline Context* as_context(ytgpu_context* h) { return reinterpret_cast<Context*>(h); }

// Serialises the calls made on one context (see Context::mu).
struct CtxLock {
    std::unique_lock<std::mutex> l;
    explicit CtxLock(ytgpu_context* h) : l(as_context(h)->mu) {}
};

// Kernel families whose launches need cudaFuncSetAttribute(MaxDynamicSharedMemorySize) on each device.
enum FuncAttrFamily : u32 { FA_SORT_PASS = 1u << 0, FA_GROUPBY = 1u << 2 };

// Reads and clears the device error word (synchronises the stream).
Status check_device_errors(Context* ctx);

}  // namespace ytgpu
