// projectultra_b200/csrc/pu_ctx.cu — context, error reporting, scratch buffers.
#include <algorithm>

#include "pu_internal.h"

namespace pu {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

pu_status Buffer::reserve(size_t bytes) {
    if (bytes <= cap) return PU_OK;
    release();
    size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = pinned_host ? cudaMallocHost(&ptr, want) : cudaMalloc(&ptr, want);
    if (e != cudaSuccess) {
        ptr = nullptr;
        cap = 0;
        set_error("allocation of %zu bytes failed: %s", want, cudaGetErrorString(e));
        return PU_ERR_NOMEM;
    }
    cap = want;
    return PU_OK;
}

void Buffer::release() {
    if (ptr) {
        if (pinned_host) cudaFreeHost(ptr);
        else cudaFree(ptr);
    }
    ptr = nullptr;
    cap = 0;
}

pu_status HostStage::run(const std::function<pu_status(size_t)>& body) {
    if (B_ == 0) return PU_OK;
    constexpr size_t kSlabBytes = size_t(64) << 20;   // staged row bytes per slab
    std::stable_sort(arrays_.begin(), arrays_.end(), [](const Array& a, const Array& b) { return a.kind < b.kind; });
    size_t row_bytes = 0;
    for (const Array& a : arrays_)
        if (a.host && a.kind != kWhole) row_bytes += a.row;
    const size_t slab = std::max<size_t>(1, std::min(B_, kSlabBytes / std::max<size_t>(row_bytes, 1)));
    // packed layout: [whole][in][inout][out]; the first slab copies from 0, later ones from the first per-row array
    size_t total = 0, rows_begin = SIZE_MAX, h2d_end = 0, d2h_begin = SIZE_MAX, out_begin = SIZE_MAX;
    for (Array& a : arrays_) {
        if (!a.host) continue;
        total = (total + 255) & ~size_t(255);
        a.off = total;
        total += a.kind == kWhole ? a.row : slab * a.row;
        if (a.kind != kWhole) rows_begin = std::min(rows_begin, a.off);
        if (a.kind != kOut) h2d_end = total;
        if (a.kind == kInOut || a.kind == kOut) d2h_begin = std::min(d2h_begin, a.off);
        if (a.kind == kOut) out_begin = std::min(out_begin, a.off);
    }
    pu_status s;
    if ((s = ctx_->stage_dev.reserve(total)) != PU_OK || (s = ctx_->stage_host.reserve(total)) != PU_OK) return s;
    char* dev = static_cast<char*>(ctx_->stage_dev.ptr);
    char* pin = static_cast<char*>(ctx_->stage_host.ptr);
    for (Array& a : arrays_) {
        a.bind(a.host ? dev + a.off : nullptr);
        if (a.host && a.kind == kWhole) std::memcpy(pin + a.off, a.host, a.row);
    }
    auto rows = [](char* dst, size_t dst_stride, const char* src, size_t src_stride, size_t row, size_t n) {
        if (dst_stride == row && src_stride == row) std::memcpy(dst, src, n * row);
        else for (size_t b = 0; b < n; ++b) std::memcpy(dst + b * dst_stride, src + b * src_stride, row);
    };
    for (size_t off = 0; off < B_; off += slab) {
        const size_t nb = std::min(slab, B_ - off);
        for (const Array& a : arrays_)
            if (a.host && (a.kind == kIn || a.kind == kInOut)) rows(pin + a.off, a.row, a.host + off * a.stride, a.stride, a.row, nb);
        const size_t h2d_begin = off == 0 ? 0 : std::min(rows_begin, h2d_end);
        if (h2d_end > h2d_begin) PU_CUDA_TRY(cudaMemcpyAsync(dev + h2d_begin, pin + h2d_begin, h2d_end - h2d_begin, cudaMemcpyHostToDevice, st_));
        if (out_begin < total) PU_CUDA_TRY(cudaMemsetAsync(dev + out_begin, 0, total - out_begin, st_));
        if ((s = body(nb)) != PU_OK) {
            cudaStreamSynchronize(st_);   // the staging buffers are reused by the next call: leave no copy in flight
            return s;
        }
        if (d2h_begin < total) PU_CUDA_TRY(cudaMemcpyAsync(pin + d2h_begin, dev + d2h_begin, total - d2h_begin, cudaMemcpyDeviceToHost, st_));
        PU_CUDA_TRY(cudaStreamSynchronize(st_));
        for (const Array& a : arrays_)
            if (a.host && (a.kind == kInOut || a.kind == kOut)) rows(a.host + off * a.stride, a.stride, pin + a.off, a.row, a.row, nb);
    }
    return PU_OK;
}

}  // namespace pu

extern "C" {

int pu_abi_version(void) { return 1; }

const char* pu_status_string(pu_status s) {
    switch (s) {
        case PU_OK: return "ok";
        case PU_ERR_INVALID: return "invalid argument";
        case PU_ERR_CUDA: return "CUDA error";
        case PU_ERR_NOMEM: return "out of memory";
        case PU_ERR_UNSUPPORTED: return "unsupported configuration";
    }
    return "unknown";
}

const char* pu_last_error(void) { return pu::g_err; }

pu_status pu_init(int device, pu_ctx** out) {
    PU_REQUIRE(out != nullptr, "pu_init: out is NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        pu::set_error("pu_init: no CUDA device (%s); this library has no CPU fallback",
                      e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
        return PU_ERR_CUDA;
    }
    PU_REQUIRE(device >= 0 && device < n, "pu_init: device index out of range");
    PU_CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    PU_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        pu::set_error("pu_init: device %d is sm_%d%d; kernels are built for sm_100a only", device, prop.major, prop.minor);
        return PU_ERR_CUDA;
    }
    pu_ctx* c = new pu_ctx();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    c->cc_major = prop.major;
    c->cc_minor = prop.minor;
    c->stage_host.pinned_host = true;
    e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        delete c;
        pu::set_error("pu_init: cudaStreamCreate failed: %s", cudaGetErrorString(e));
        return PU_ERR_CUDA;
    }
    for (auto& sl : c->pipe) {
        sl.h_in.pinned_host = true;
        sl.h_out.pinned_host = true;
        if (cudaStreamCreateWithFlags(&sl.stream, cudaStreamNonBlocking) != cudaSuccess) sl.stream = nullptr;
    }
    if (cudaEventCreateWithFlags(&c->pipe_ev, cudaEventDisableTiming) != cudaSuccess) c->pipe_ev = nullptr;
    if (!c->pipe[0].stream || !c->pipe[1].stream || !c->pipe_ev) {
        pu::set_error("pu_init: could not create the pipeline streams");
        pu_destroy(c);
        return PU_ERR_CUDA;
    }
    *out = c;
    return PU_OK;
}

void pu_destroy(pu_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    c->stage_dev.release();
    c->stage_host.release();
    c->d_aux.release();
    c->f_bytes.release(); c->f_ok.release(); c->f_iters.release();
    for (auto& sl : c->pipe) {
        if (sl.stream) cudaStreamSynchronize(sl.stream);
        sl.d_in.release(); sl.d_llr.release(); sl.d_out.release(); sl.h_in.release(); sl.h_out.release();
        if (sl.stream) cudaStreamDestroy(sl.stream);
    }
    if (c->pipe_ev) cudaEventDestroy(c->pipe_ev);
    c->cfo_mix.release();
    for (auto& b : c->sweep) b.release();
    for (auto& e : c->sweep_ev) if (e) cudaEventDestroy(e);
    cudaStreamDestroy(c->stream);
    delete c;
}

int pu_device_sm_count(const pu_ctx* c) { return c ? c->sm_count : 0; }

pu_status pu_synchronize(pu_ctx* c, void* stream) {
    PU_REQUIRE(c != nullptr, "pu_synchronize: ctx is NULL");
    PU_CUDA_TRY(cudaStreamSynchronize(pu::pick_stream(c, stream)));
    return PU_OK;
}

uint64_t pu_kernel_launches(const pu_ctx* c) { return c ? c->launches.load() : 0; }

void pu_transfer_bytes(const pu_ctx* c, uint64_t* h2d, uint64_t* d2h) {
    if (h2d) *h2d = c ? c->h2d_bytes.load() : 0;
    if (d2h) *d2h = c ? c->d2h_bytes.load() : 0;
}

}  // extern "C"
