// fp32 vector helpers behind the reference's device BLAS-ish entry points
// (blas.h:43-53 fill/copy/axpy/scal_ongpu, activations.h:18 activate_array_ongpu).  They are not on
// the detection hot path (the forward pass fuses all of this into the convolution epilogues); they
// exist so callers that touch cuda_make_array buffers directly keep linking.  HBM-bound grid-stride
// kernels; unit-stride calls move float4s.
#include "y2_common.cuh"

namespace y2 {

static inline int vec_grid(long long n, int threads)
{
    long long blocks = (n + threads - 1) / threads;
    const long long cap = (long long)sm_count() * 16;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}

enum { OP_FILL = 0, OP_COPY = 1, OP_AXPY = 2, OP_SCAL = 3 };

template <int OP>
__global__ void vec_op_kernel(long long n, float alpha, const float *__restrict__ x, long long incx,
                              float *__restrict__ y, long long incy)
{
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x) {
        float *py = y + i * incy;
        if (OP == OP_FILL) *py = alpha;
        else if (OP == OP_COPY) *py = x[i * incx];
        else if (OP == OP_AXPY) *py = __fadd_rn(*py, __fmul_rn(alpha, x[i * incx])); // Y[i] += ALPHA*X[i], no fma
        else *py = __fmul_rn(*py, alpha);
    }
}

template <int OP>
__global__ void vec_op4_kernel(long long n4, float alpha, const float4 *__restrict__ x, float4 *__restrict__ y)
{
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4;
         i += (long long)gridDim.x * blockDim.x) {
        float4 v;
        if (OP == OP_FILL) v = make_float4(alpha, alpha, alpha, alpha);
        else if (OP == OP_COPY) v = x[i];
        else if (OP == OP_AXPY) {
            const float4 a = x[i];
            v = y[i];
            v.x = __fadd_rn(v.x, __fmul_rn(alpha, a.x));
            v.y = __fadd_rn(v.y, __fmul_rn(alpha, a.y));
            v.z = __fadd_rn(v.z, __fmul_rn(alpha, a.z));
            v.w = __fadd_rn(v.w, __fmul_rn(alpha, a.w));
        } else {
            v = y[i];
            v.x = __fmul_rn(v.x, alpha);
            v.y = __fmul_rn(v.y, alpha);
            v.z = __fmul_rn(v.z, alpha);
            v.w = __fmul_rn(v.w, alpha);
        }
        y[i] = v;
    }
}

// ACTIVATION numbering of activations.h:6-8:
// LOGISTIC, RELU, RELIE, LINEAR, RAMP, TANH, PLSE, LEAKY, ELU, LOGGY, STAIR, HARDTAN, LHTAN
__device__ __forceinline__ float activate(float x, int a)
{
    switch (a) {
    case 0: return 1.f / (1.f + expf(-x));
    case 1: return x > 0.f ? x : 0.f;
    case 2: return x > 0.f ? x : .01f * x;
    case 3: return x;
    case 4: return (x > 0.f ? x : 0.f) + .1f * x;
    case 5: return tanhf(x); /* = 2/(1+e^-2x) - 1, which keeps only a few bits for |x| << 1 */
    case 6: return x < -4.f ? .01f * (x + 4.f) : x > 4.f ? .01f * (x - 4.f) + 1.f : .125f * x + .5f;
    case 7: return x > 0.f ? x : .1f * x;
    case 8: return x >= 0.f ? x : expm1f(x);
    case 9: return tanhf(.5f * x); /* = 2/(1+e^-x) - 1 */
    case 10: {
        /* floor(x / 2.) of the reference, in double there: floor(floor(x) / 2), x / 2.f would underflow to -0
         * for the smallest negative denormal */
        const int n = (int)floorf(x);
        const float half = (float)(n >> 1);
        return (n % 2 == 0) ? half : (x - n) + half;
    }
    case 11: return x < -1.f ? -1.f : x > 1.f ? 1.f : x;
    case 12: return x < 0.f ? .001f * x : x > 1.f ? .001f * (x - 1.f) + 1.f : x;
    }
    return x;
}

__global__ void vec_activate_kernel(float *__restrict__ x, long long n, int a)
{
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x)
        x[i] = activate(x[i], a);
}

// ---- gemm_ongpu / im2col_ongpu of the helper surface (gemm.c:173-183, im2col_kernels.cu:48-61) -----------------
// Plain fp32 CUDA-core kernels for callers that still link these names (the reference's layer code around the hot
// path: connected / rnn training utilities, test_gpu_blas).  The network's own convolutions never come here: they are
// implicit GEMMs on the tensor cores.  C (row-major M x N) = ALPHA * op(A) * op(B) + BETA * C.
template <int TA, int TB>
__global__ void sgemm_kernel(int M, int N, int K, float alpha, const float *__restrict__ A, int lda,
                             const float *__restrict__ B, int ldb, float beta, float *__restrict__ C, int ldc)
{
    __shared__ float sa[32][33], sb[32][33];
    const int tx = threadIdx.x, ty = threadIdx.y;  // 32 x 8
    const int row0 = blockIdx.y * 32, col0 = blockIdx.x * 32;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int k0 = 0; k0 < K; k0 += 32) {
        for (int r = ty; r < 32; r += 8) {
            const int i = row0 + r, k = k0 + tx;  // sa[r][tx] = op(A)[i][k]
            sa[r][tx] = (i < M && k < K) ? (TA ? A[(size_t)k * lda + i] : A[(size_t)i * lda + k]) : 0.f;
            const int kb = k0 + r, j = col0 + tx;  // sb[r][tx] = op(B)[kb][j]
            sb[r][tx] = (kb < K && j < N) ? (TB ? B[(size_t)j * ldb + kb] : B[(size_t)kb * ldb + j]) : 0.f;
        }
        __syncthreads();
#pragma unroll 8
        for (int k = 0; k < 32; ++k) {
            const float b = sb[k][tx];
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[q] = fmaf(sa[ty + 8 * q][k], b, acc[q]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int i = row0 + ty + 8 * q, j = col0 + tx;
        if (i < M && j < N) {
            float *c = C + (size_t)i * ldc + j;
            *c = alpha * acc[q] + (beta == 0.f ? 0.f : beta * *c);
        }
    }
}

// col[(c*k*k + i*k + j)][h_out][w_out] = im[c][h_out*stride - pad + i][w_out*stride - pad + j], 0 outside
__global__ void im2col_kernel(const float *__restrict__ im, int channels, int height, int width, int ksize, int stride,
                              int pad, int height_col, int width_col, float *__restrict__ col)
{
    const long long total = (long long)channels * ksize * ksize * height_col * width_col;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        const int w_out = (int)(t % width_col);
        const int h_out = (int)((t / width_col) % height_col);
        const int row = (int)(t / ((long long)width_col * height_col));
        const int j = row % ksize, i = (row / ksize) % ksize, c = row / (ksize * ksize);
        const int h = h_out * stride - pad + i, w = w_out * stride - pad + j;
        col[t] = (h >= 0 && w >= 0 && h < height && w < width) ? im[((size_t)c * height + h) * width + w] : 0.f;
    }
}

template <int OP>
static int vec_launch(long long n, float alpha, const float *x, long long incx, float *y, long long incy,
                      y2_stream_t s)
{
    if (n <= 0) return Y2_OK;
    if (!y || (OP != OP_FILL && OP != OP_SCAL && !x)) {
        set_error("y2_vec_*: null vector");
        return Y2_EINVAL;
    }
    const bool unit = incy == 1 && (OP == OP_FILL || OP == OP_SCAL || incx == 1);
    const bool aligned = ((uintptr_t)y % 16 == 0) && (OP == OP_FILL || OP == OP_SCAL || (uintptr_t)x % 16 == 0);
    const long long n4 = (unit && aligned) ? n / 4 : 0;
    if (n4)
        vec_op4_kernel<OP><<<vec_grid(n4, 256), 256, 0, to_stream(s)>>>(n4, alpha, (const float4 *)x, (float4 *)y);
    if (n > n4 * 4)
        vec_op_kernel<OP><<<vec_grid(n - n4 * 4, 256), 256, 0, to_stream(s)>>>(
            n - n4 * 4, alpha, x ? x + n4 * 4 * incx : x, incx, y + n4 * 4 * incy, incy);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

} // namespace y2

using namespace y2;

extern "C" int y2_vec_fill(long long n, float alpha, float *x, long long incx, y2_stream_t s)
{
    return vec_launch<OP_FILL>(n, alpha, nullptr, 1, x, incx, s);
}

extern "C" int y2_vec_copy(long long n, const float *x, long long incx, float *y, long long incy, y2_stream_t s)
{
    return vec_launch<OP_COPY>(n, 0.f, x, incx, y, incy, s);
}

extern "C" int y2_vec_axpy(long long n, float alpha, const float *x, long long incx, float *y, long long incy,
                           y2_stream_t s)
{
    return vec_launch<OP_AXPY>(n, alpha, x, incx, y, incy, s);
}

extern "C" int y2_vec_scal(long long n, float alpha, float *x, long long incx, y2_stream_t s)
{
    return vec_launch<OP_SCAL>(n, alpha, nullptr, 1, x, incx, s);
}

extern "C" int y2_vec_activate(float *x, long long n, int activation, y2_stream_t s)
{
    if (n <= 0) return Y2_OK;
    if (!x || activation < 0 || activation > 12) {
        set_error("y2_vec_activate: invalid arguments (activation=%d)", activation);
        return Y2_EINVAL;
    }
    vec_activate_kernel<<<vec_grid(n, 256), 256, 0, to_stream(s)>>>(x, n, activation);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_sgemm(int TA, int TB, int M, int N, int K, float alpha, const float *A, int lda, const float *B,
                        int ldb, float beta, float *C, int ldc, y2_stream_t s)
{
    if (M <= 0 || N <= 0) return Y2_OK;
    if (!A || !B || !C || K < 0) return Y2_EINVAL;
    const dim3 grid((unsigned)((N + 31) / 32), (unsigned)((M + 31) / 32)), block(32, 8);
    if (!TA && !TB) sgemm_kernel<0, 0><<<grid, block, 0, to_stream(s)>>>(M, N, K, alpha, A, lda, B, ldb, beta, C, ldc);
    else if (TA && !TB) sgemm_kernel<1, 0><<<grid, block, 0, to_stream(s)>>>(M, N, K, alpha, A, lda, B, ldb, beta, C, ldc);
    else if (!TA && TB) sgemm_kernel<0, 1><<<grid, block, 0, to_stream(s)>>>(M, N, K, alpha, A, lda, B, ldb, beta, C, ldc);
    else sgemm_kernel<1, 1><<<grid, block, 0, to_stream(s)>>>(M, N, K, alpha, A, lda, B, ldb, beta, C, ldc);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_im2col_f32(const float *im, int channels, int height, int width, int ksize, int stride, int pad,
                             float *col, y2_stream_t s)
{
    if (!im || !col || channels <= 0 || ksize <= 0 || stride <= 0) return Y2_EINVAL;
    const int height_col = (height + 2 * pad - ksize) / stride + 1;
    const int width_col = (width + 2 * pad - ksize) / stride + 1;
    if (height_col <= 0 || width_col <= 0) return Y2_EINVAL;
    const long long total = (long long)channels * ksize * ksize * height_col * width_col;
    im2col_kernel<<<vec_grid(total, 256), 256, 0, to_stream(s)>>>(im, channels, height, width, ksize, stride, pad,
                                                                  height_col, width_col, col);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}
