// The double instantiations of the CUDA-core kernels (stb_layer.dtype == STB_F64): the layer kernel
// (generic_tile.cuh), the parameter-free layers and the element-wise backward (backward_tile.cuh).
// They live in a translation unit of their own so the fp32 objects stay as they are.  The spline
// constants are the reference's double values (stb_math.cuh: RqsDefaultsT / CubDefaultsT<double>).
#include "backward_tile.cuh"
#include "generic_tile.cuh"

namespace stb {

template <int KIND>
__global__ void __launch_bounds__(kGenThreads) generic_layer_f64_kernel(const GenArgs A) {
    generic_layer_tile<double, KIND>(A, DefaultOpts<KIND, double>(), threadIdx.x);
}

template <int KIND>
__global__ void __launch_bounds__(kGenThreads) generic_layer_opts_f64_kernel(const GenArgs A,
                                                                             const SplineOptsT<double> o) {
    generic_layer_tile<double, KIND>(A, o, threadIdx.x);
}

__global__ void pointwise_f64_kernel(int kind, int direction, const double* __restrict__ x, double* __restrict__ y,
                                     const int32_t* __restrict__ perm, double* __restrict__ ldj, int ldj_mode,
                                     int base_log_prob, int d, long long rows) {
    pointwise_row<double>(kind, direction, x, y, perm, ldj, ldj_mode, base_log_prob, d, rows);
}

template <int KIND>
__global__ void __launch_bounds__(kBThreads) elementwise_backward_f64_kernel(const BwdArgs A) {
    elementwise_backward_tile<double, KIND>(A, DefaultOpts<KIND, double>(), threadIdx.x);
}

template <int KIND>
__global__ void __launch_bounds__(kBThreads) elementwise_backward_opts_f64_kernel(const BwdArgs A,
                                                                                  const SplineOptsT<double> o) {
    elementwise_backward_tile<double, KIND>(A, o, threadIdx.x);
}

int generic_layer_launch_f64(const stb_layer* L, const GenArgs& A, size_t smem, unsigned tiles, cudaStream_t stream) {
    const char* name = "generic_layer_f64_kernel";
    if (L->spline.custom && (L->kind == STB_RQS || L->kind == STB_CUBIC)) {
        const SplineOptsT<double> o = make_spline_opts<SplineOptsT<double>>(L->spline);
        return L->kind == STB_RQS
                   ? launch_kernel(generic_layer_opts_f64_kernel<STB_RQS>, tiles, kGenThreads, smem, stream, name, A, o)
                   : launch_kernel(generic_layer_opts_f64_kernel<STB_CUBIC>, tiles, kGenThreads, smem, stream, name, A, o);
    }
    switch (L->kind) {
        case STB_AFFINE: return launch_kernel(generic_layer_f64_kernel<STB_AFFINE>, tiles, kGenThreads, smem, stream, name, A);
        case STB_RQS: return launch_kernel(generic_layer_f64_kernel<STB_RQS>, tiles, kGenThreads, smem, stream, name, A);
        case STB_CUBIC: return launch_kernel(generic_layer_f64_kernel<STB_CUBIC>, tiles, kGenThreads, smem, stream, name, A);
        default: return launch_kernel(generic_layer_f64_kernel<STB_CONT_AFFINE>, tiles, kGenThreads, smem, stream, name, A);
    }
}

int pointwise_launch_f64(int kind, int direction, const float* x, float* y, const int32_t* perm, float* ldj,
                         int ldj_mode, int base_log_prob, int d, long long rows, unsigned blocks, int threads,
                         cudaStream_t stream) {
    return launch_kernel(pointwise_f64_kernel, blocks, threads, 0, stream, "pointwise_f64_kernel", kind, direction,
                         reinterpret_cast<const double*>(x), reinterpret_cast<double*>(y), perm,
                         reinterpret_cast<double*>(ldj), ldj_mode, base_log_prob, d, rows);
}

int elementwise_backward_launch_f64(const stb_layer* L, const BwdArgs& A, size_t smem, unsigned tiles,
                                    cudaStream_t stream) {
    const char* name = "elementwise_backward_f64_kernel";
    if (L->spline.custom && (L->kind == STB_RQS || L->kind == STB_CUBIC)) {
        const SplineOptsT<double> o = make_spline_opts<SplineOptsT<double>>(L->spline);
        return L->kind == STB_RQS
                   ? launch_kernel(elementwise_backward_opts_f64_kernel<STB_RQS>, tiles, kBThreads, smem, stream, name, A, o)
                   : launch_kernel(elementwise_backward_opts_f64_kernel<STB_CUBIC>, tiles, kBThreads, smem, stream, name, A, o);
    }
    switch (L->kind) {
        case STB_AFFINE: return launch_kernel(elementwise_backward_f64_kernel<STB_AFFINE>, tiles, kBThreads, smem, stream, name, A);
        case STB_RQS: return launch_kernel(elementwise_backward_f64_kernel<STB_RQS>, tiles, kBThreads, smem, stream, name, A);
        default: return launch_kernel(elementwise_backward_f64_kernel<STB_CUBIC>, tiles, kBThreads, smem, stream, name, A);
    }
}

}  // namespace stb
