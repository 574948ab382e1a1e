// projectultra_b200/csrc/refmath_eval.cu — evaluates the libm restatements of ref_math.cuh on the host or on the
// device over arrays, so tests can pin them against the host libm (CPU) and check device == host (GPU).
#include "pu_internal.h"
#include "ref_math.cuh"

namespace pu {

PU_RM float refmath_apply(int op, float a, float b) {
    switch (op) {
        case 0: return refmath::atan2f_ref(a, b);
        case 1: return refmath::sinf_ref(a);
        case 2: return refmath::cosf_ref(a);
        case 3: return refmath::hypotf_ref(a, b);
        default: return refmath::atanf_ref(a);
    }
}

__global__ void refmath_kernel(int op, const float* a, const float* b, float* out, size_t n) {
    const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
    if (i < n) out[i] = refmath_apply(op, a[i], b ? b[i] : 0.0f);
}

}  // namespace pu

extern "C" pu_status pu_refmath_eval(pu_ctx* ctx, int op, const float* a, const float* b, float* out, size_t n) {
    PU_REQUIRE(a && out, "pu_refmath_eval: NULL argument");
    if (!ctx) {   // host evaluation
        for (size_t i = 0; i < n; ++i) out[i] = pu::refmath_apply(op, a[i], b ? b[i] : 0.0f);
        return PU_OK;
    }
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    pu::HostStage hs(ctx, ctx->stream, n);
    const float *da, *db;
    float* dout;
    hs.in(&da, a, 1);
    hs.in(&db, b, 1);
    hs.out(&dout, out, 1);
    return hs.run([&](size_t nb) -> pu_status {
        pu::refmath_kernel<<<static_cast<unsigned>((nb + 255) / 256), 256, 0, ctx->stream>>>(op, da, db, dout, nb);
        ctx->launches.fetch_add(1);
        PU_CUDA_TRY(cudaGetLastError());
        return PU_OK;
    });
}
