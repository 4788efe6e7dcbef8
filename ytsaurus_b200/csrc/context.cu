// context.cu — context lifetime, status plumbing, timers.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <new>

#include "context.cuh"

namespace ytgpu {

Status make_status(int code, const char* fmt, ...) {
    Status s;
    s.code = code;
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(s.msg, sizeof(s.msg), fmt, ap);
    va_end(ap);
    return s;
}

Status cuda_status(cudaError_t e, const char* what) {
    Status s;
    s.code = YTGPU_ERR_CUDA;
    s.cuda = (int)e;
    snprintf(s.msg, sizeof(s.msg), "%s: %s", what, cudaGetErrorString(e));
    cudaGetLastError();
    return s;
}

void Context::collect_timers() {
    if (spans.empty()) return;
    cudaStreamSynchronize(stream);
    for (auto& sp : spans) {
        float f = 0;
        if (cudaEventElapsedTime(&f, sp.start, sp.stop) == cudaSuccess) {
            if (sp.cls == KC_RADIX_PASS) pass_ms.push_back(f);
            else ms[sp.cls] += f;
        }
        cudaEventDestroy(sp.start);
        cudaEventDestroy(sp.stop);
    }
    spans.clear();
}

Status check_device_errors(Context* ctx) {
    YTGPU_CUDA_TRY(cudaMemcpyAsync(ctx->host_err, ctx->dev_err, 4, cudaMemcpyDeviceToHost, ctx->stream));
    YTGPU_CUDA_TRY(cudaMemsetAsync(ctx->dev_err, 0, 4, ctx->stream));
    YTGPU_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    u32 e = *ctx->host_err;
    if (e == 0) return Status{};
    if (e & DE_UNSUPPORTED_TYPE)
        return make_status(YTGPU_ERR_UNSUPPORTED, "key column holds an Any/Composite value: YSON comparison is not available on the GPU path");
    if (e & DE_SCHEMA_VIOLATION)
        return make_status(YTGPU_ERR_SCHEMA_VIOLATION, "a key value's type differs from the declared key column type");
    if (e & DE_STRING_TOO_LONG)
        return make_status(YTGPU_ERR_SCHEMA_VIOLATION, "a key string is longer than the declared key column width");
    if (e & DE_PART_BAD_TYPE)
        return make_status(YTGPU_ERR_PARTITION_BAD_TYPE, "Invalid partition column value type: expected type \"int64\" or \"uint64\"");
    if (e & DE_PART_NEGATIVE) return make_status(YTGPU_ERR_PARTITION_NEGATIVE, "Received negative partition index");
    if (e & DE_PART_OUT_OF_BOUNDS) return make_status(YTGPU_ERR_PARTITION_OUT_OF_BOUNDS, "Partition index is out of bounds");
    if (e & DE_PART_NO_COLUMN) return make_status(YTGPU_ERR_PARTITION_NO_COLUMN, "Row does not contain partition column");
    if (e & DE_TABLE_FULL) return make_status(YTGPU_ERR_INVALID_ARGUMENT, "group-by hash table capacity exceeded");
    if (e & DE_PEER_TIMEOUT)
        return make_status(YTGPU_ERR_CUDA, "in-box shuffle: a peer GPU did not reach the barrier within 20 s (a rank failed or never made the call)");
    if (e & DE_BAD_PARTITION_INDEX)
        return make_status(YTGPU_ERR_INVALID_ARGUMENT, "partition index outside [0, partition_count) or partition row counts that disagree with it");
    return make_status(YTGPU_ERR_CUDA, "unknown device error word 0x%x", e);
}

}  // namespace ytgpu

using namespace ytgpu;

extern "C" {

int ytgpu_abi_version(void) { return YTGPU_ABI_VERSION; }

int ytgpu_context_create(int device, void* cuda_stream, ytgpu_context** out, ytgpu_error* err) {
    if (!out) return fill_error(err, make_status(YTGPU_ERR_INVALID_ARGUMENT, "out is null"));
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        cudaGetLastError();
        return fill_error(err, make_status(YTGPU_ERR_CUDA, "no CUDA device available (%s); this library has no CPU fallback",
                                         cudaGetErrorString(e)));
    }
    if (device < 0 || device >= count)
        return fill_error(err, make_status(YTGPU_ERR_INVALID_ARGUMENT, "device %d out of range [0, %d)", device, count));
    if ((e = cudaSetDevice(device)) != cudaSuccess) return fill_error(err, cuda_status(e, "cudaSetDevice"));
    Context* c = new (std::nothrow) Context();
    if (!c) return fill_error(err, make_status(YTGPU_ERR_OUT_OF_MEMORY, "host allocation failed"));
    c->device = device;
    if (cuda_stream) {
        c->stream = static_cast<cudaStream_t>(cuda_stream);
    } else {
        if ((e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)) != cudaSuccess) {
            delete c;
            return fill_error(err, cuda_status(e, "cudaStreamCreate"));
        }
        c->owns_stream = true;
    }
    // keep freed scratch cached in the stream-ordered pool between calls
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        uint64_t thr = UINT64_MAX;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    if ((e = cudaMalloc(&c->dev_err, 4)) != cudaSuccess || (e = cudaMemset(c->dev_err, 0, 4)) != cudaSuccess ||
        (e = cudaHostAlloc(&c->host_err, 16, cudaHostAllocDefault)) != cudaSuccess) {
        Status s = cuda_status(e, "context allocation");
        delete c;
        return fill_error(err, s);
    }
    c->host_err[0] = c->host_err[1] = c->host_err[2] = c->host_err[3] = 0;
    *out = reinterpret_cast<ytgpu_context*>(c);
    return fill_error(err, Status{});
}

void ytgpu_context_destroy(ytgpu_context* h) {
    if (!h) return;
    Context* c = reinterpret_cast<Context*>(h);
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    c->collect_timers();
    if (c->dev_err) cudaFree(c->dev_err);
    if (c->host_err) cudaFreeHost(c->host_err);
    if (c->owns_stream) cudaStreamDestroy(c->stream);
    delete c;
}

int ytgpu_context_synchronize(ytgpu_context* h, ytgpu_error* err) {
    Context* c = reinterpret_cast<Context*>(h);
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) return fill_error(err, cuda_status(e, "cudaStreamSynchronize"));
    return fill_error(err, Status{});
}

uint64_t ytgpu_context_launch_count(const ytgpu_context* h) { return reinterpret_cast<const Context*>(h)->launches; }

double ytgpu_context_kernel_ms(ytgpu_context* h, int which, uint64_t* launches) {
    Context* c = reinterpret_cast<Context*>(h);
    if (which < 0 || which >= KC_COUNT) return 0.0;
    c->collect_timers();
    if (which == KC_RADIX_PASS || which == KC_PASS_SKIPPED) {
        // Pass launches are timed one by one; launches of skipped digits exit at once.  A launch counts as "active"
        // when it ran at least a fifth as long as the longest one.
        float mx = 0;
        for (float f : c->pass_ms) mx = f > mx ? f : mx;
        double act = 0, skip = 0;
        uint64_t nact = 0, nskip = 0;
        for (float f : c->pass_ms) {
            if (f >= 0.2f * mx) { act += f; ++nact; } else { skip += f; ++nskip; }
        }
        if (launches) *launches = which == KC_RADIX_PASS ? nact : nskip;
        return which == KC_RADIX_PASS ? act : skip;
    }
    if (launches) *launches = c->timed_launches[which];
    return c->ms[which];
}

void ytgpu_context_reset_timers(ytgpu_context* h) {
    Context* c = reinterpret_cast<Context*>(h);
    c->collect_timers();
    c->pass_ms.clear();
    for (int i = 0; i < KC_COUNT; ++i) {
        c->ms[i] = 0;
        c->timed_launches[i] = 0;
    }
}

uint64_t ytgpu_context_last_sort_passes(ytgpu_context* h) {
    Context* c = reinterpret_cast<Context*>(h);
    cudaStreamSynchronize(c->stream);
    return c->host_err[1] + (c->host_err[3] ? c->host_err[2] : 0);
}

int ytgpu_context_set_option(ytgpu_context* h, const char* name, int64_t value, ytgpu_error* err) {
    if (!h || !name) return fill_error(err, make_status(YTGPU_ERR_INVALID_ARGUMENT, "null argument"));
    CtxLock lock(h);
    Context* c = reinterpret_cast<Context*>(h);
    if (strcmp(name, "sort_hybrid") == 0) {
        c->opt_sort_hybrid = value ? 1 : 0;
        return fill_error(err, Status{});
    }
    if (strcmp(name, "merge_path") == 0) {
        c->opt_merge_path = value ? 1 : 0;
        return fill_error(err, Status{});
    }
    return fill_error(err, make_status(YTGPU_ERR_INVALID_ARGUMENT, "unknown option '%s'", name));
}

int ytgpu_context_get_option(ytgpu_context* h, const char* name, int64_t* value, ytgpu_error* err) {
    if (!h || !name || !value) return fill_error(err, make_status(YTGPU_ERR_INVALID_ARGUMENT, "null argument"));
    CtxLock lock(h);
    Context* c = reinterpret_cast<Context*>(h);
    if (strcmp(name, "sort_hybrid") == 0) *value = c->opt_sort_hybrid;
    else if (strcmp(name, "merge_path") == 0) *value = c->opt_merge_path;
    else if (strcmp(name, "last_merge_used_merge_path") == 0) *value = c->last_merge_used_merge_path ? 1 : 0;
    else return fill_error(err, make_status(YTGPU_ERR_INVALID_ARGUMENT, "unknown option '%s'", name));
    return fill_error(err, Status{});
}

void ytgpu_context_enable_timers(ytgpu_context* h, int enabled) {
    reinterpret_cast<Context*>(h)->timers_enabled = enabled != 0;
}

int ytgpu_context_notify(ytgpu_context* h, ytgpu_callback fn, void* user, ytgpu_error* err) {
    if (!h || !fn) return fill_error(err, make_status(YTGPU_ERR_INVALID_ARGUMENT, "null argument"));
    CtxLock lock(h);
    Context* c = reinterpret_cast<Context*>(h);
    cudaError_t e = cudaSetDevice(c->device);
    if (e == cudaSuccess) e = cudaLaunchHostFunc(c->stream, fn, user);
    if (e != cudaSuccess) return fill_error(err, cuda_status(e, "cudaLaunchHostFunc"));
    return fill_error(err, Status{});
}

void* ytgpu_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}

void ytgpu_host_free(void* p) {
    if (p) cudaFreeHost(p);
}

}  // extern "C"
