// Gated-GELU feed-forward of T5 v1.1 / Flan-T5 (T5DenseGatedActDense, HF/models/t5/modeling_t5.py:106-132), the elementwise
// half: the two input projections x wi_0^T | x wi_1^T come out of ONE GEMM against the concatenated [wi_0; wi_1] operand, so
// row m of u [M, 2 d_ff] holds a = u[m, 0:d_ff] and b = u[m, d_ff:2 d_ff].
//   fwd  h  = dropout(gelu_new(a) * b)                                  [M, d_ff]
//   bwd  du = [dh' * b * gelu_new'(a) | dh' * gelu_new(a)],  dh' = dropout(dh)   [M, 2 d_ff]
// gelu_new is the tanh form, 0.5 x (1 + tanh(sqrt(2/pi) (x + 0.044715 x^3))) (HF/activations.py NewGELUActivation), not the
// erf GELU of Swin.  The dropout mask is the one klab_dropout_apply draws for a contiguous [M, d_ff] tensor with the same
// (p, seed, *seed_ptr): element (m, j) has counter index m * d_ff + j, so backward regenerates it and a CUDA-graph replay after
// klab_seed_advance draws a fresh one.
//
// Pure bandwidth: one thread handles 8 consecutive columns of one row (16-byte loads and stores for bf16, two per operand for
// fp32), fp32 arithmetic throughout.  d_ff must be a multiple of 8 and the tensors contiguous and 16-byte aligned.
#include "common.cuh"

namespace klab {
void count_launch(int n = 1);
namespace {

constexpr int GEGLU_THREADS = 256;
constexpr float GELU_K0 = 0.7978845608028654f;             // sqrt(2 / pi)
constexpr float GELU_K1 = 0.044715f;

__device__ __forceinline__ void gelu_new_and_grad(float x, float& g, float& dg) {
    const float x2 = x * x;
    const float t = tanhf(GELU_K0 * (x + GELU_K1 * x2 * x));
    g = 0.5f * x * (1.0f + t);
    dg = 0.5f * (1.0f + t) + 0.5f * x * (1.0f - t * t) * GELU_K0 * (1.0f + 3.0f * GELU_K1 * x2);
}

__device__ __forceinline__ float gelu_new(float x) {
    return 0.5f * x * (1.0f + tanhf(GELU_K0 * (x + GELU_K1 * x * x * x)));
}

// 8 consecutive elements <-> fp32 registers
__device__ __forceinline__ void load8(const __nv_bfloat16* p, float (&v)[8]) {
    const uint4 q = *reinterpret_cast<const uint4*>(p);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&q);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 f = __bfloat1622float2(h[i]);
        v[2 * i] = f.x;
        v[2 * i + 1] = f.y;
    }
}
__device__ __forceinline__ void load8(const float* p, float (&v)[8]) {
    const float4 a = reinterpret_cast<const float4*>(p)[0], b = reinterpret_cast<const float4*>(p)[1];
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
    v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void store8(__nv_bfloat16* p, const float (&v)[8]) {
    uint4 q;
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&q);
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
    *reinterpret_cast<uint4*>(p) = q;
}
__device__ __forceinline__ void store8(float* p, const float (&v)[8]) {
    reinterpret_cast<float4*>(p)[0] = make_float4(v[0], v[1], v[2], v[3]);
    reinterpret_cast<float4*>(p)[1] = make_float4(v[4], v[5], v[6], v[7]);
}

template <typename T>
__global__ void __launch_bounds__(GEGLU_THREADS) geglu_fwd_kernel(const T* __restrict__ u, T* __restrict__ h, long long n8, int dff8,
                                                                  unsigned long long seed, const unsigned long long* __restrict__ seed_ptr,
                                                                  float p) {
    if (seed_ptr) seed += *seed_ptr;
    const DropKey key = make_drop_key(seed, p);
    const long long dff = 8ll * dff8;
    const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n8; i += stride) {
        const long long m = i / dff8;
        const long long j = 8ll * (i - m * dff8);
        const T* row = u + 2 * dff * m;
        float a[8], b[8];
        load8(row + j, a);
        load8(row + dff + j, b);
#pragma unroll
        for (int e = 0; e < 8; ++e) a[e] = gelu_new(a[e]) * b[e];
        if (key.on) dropout_apply_run<8>(key, static_cast<uint64_t>(m * dff + j), a);
        store8(h + m * dff + j, a);
    }
}

template <typename T>
__global__ void __launch_bounds__(GEGLU_THREADS) geglu_bwd_kernel(const T* __restrict__ dh, const T* __restrict__ u, T* __restrict__ du,
                                                                  long long n8, int dff8, unsigned long long seed,
                                                                  const unsigned long long* __restrict__ seed_ptr, float p) {
    if (seed_ptr) seed += *seed_ptr;
    const DropKey key = make_drop_key(seed, p);
    const long long dff = 8ll * dff8;
    const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n8; i += stride) {
        const long long m = i / dff8;
        const long long j = 8ll * (i - m * dff8);
        const T* row = u + 2 * dff * m;
        float a[8], b[8], g[8];
        load8(row + j, a);
        load8(row + dff + j, b);
        load8(dh + m * dff + j, g);
        if (key.on) dropout_apply_run<8>(key, static_cast<uint64_t>(m * dff + j), g);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            float ge, dge;
            gelu_new_and_grad(a[e], ge, dge);
            a[e] = g[e] * b[e] * dge;                      // d / da
            b[e] = g[e] * ge;                              // d / db
        }
        T* out = du + 2 * dff * m;
        store8(out + j, a);
        store8(out + dff + j, b);
    }
}

unsigned geglu_grid(long long n8) {
    long long g = (n8 + GEGLU_THREADS - 1) / GEGLU_THREADS;
    const long long cap = 32ll * sm_count();
    return static_cast<unsigned>(g > cap ? cap : (g < 1 ? 1 : g));
}

int geglu_check(const char* what, int dtype, long long rows, int d_ff, float p, std::initializer_list<const void*> ptrs) {
    KLAB_REQUIRE(dtype == KLAB_BF16 || dtype == KLAB_F32, "%s: dtype %d is neither bf16 nor fp32", what, dtype);
    KLAB_REQUIRE(rows > 0 && d_ff > 0 && p >= 0.0f && p < 1.0f, "%s: bad arguments rows=%lld d_ff=%d p=%f", what, rows, d_ff, p);
    KLAB_REQUIRE(d_ff % 8 == 0, "%s: d_ff=%d must be a multiple of 8 (8 columns per thread, 16-byte vectors)", what, d_ff);
    for (const void* q : ptrs)
        KLAB_REQUIRE(q != nullptr && (reinterpret_cast<uintptr_t>(q) & 15) == 0, "%s: tensors must be 16-byte aligned", what);
    return KLAB_OK;
}

}  // namespace
}  // namespace klab

using namespace klab;

extern "C" {

int klab_geglu_fwd(void* stream, int dtype, long long rows, int d_ff, const void* u, void* h, float p, unsigned long long seed,
                   const unsigned long long* seed_ptr) {
    if (int rc = klab_check_device()) return rc;
    if (int rc = geglu_check("geglu_fwd", dtype, rows, d_ff, p, {u, h})) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const long long n8 = rows * (d_ff / 8);
    if (dtype == KLAB_BF16)
        geglu_fwd_kernel<__nv_bfloat16><<<geglu_grid(n8), GEGLU_THREADS, 0, st>>>(
            static_cast<const __nv_bfloat16*>(u), static_cast<__nv_bfloat16*>(h), n8, d_ff / 8, seed, seed_ptr, p);
    else
        geglu_fwd_kernel<float><<<geglu_grid(n8), GEGLU_THREADS, 0, st>>>(static_cast<const float*>(u), static_cast<float*>(h), n8,
                                                                          d_ff / 8, seed, seed_ptr, p);
    KLAB_LAUNCH_CHECK();
    count_launch();
    return KLAB_OK;
}

int klab_geglu_bwd(void* stream, int dtype, long long rows, int d_ff, const void* dh, const void* u, void* du, float p,
                   unsigned long long seed, const unsigned long long* seed_ptr) {
    if (int rc = klab_check_device()) return rc;
    if (int rc = geglu_check("geglu_bwd", dtype, rows, d_ff, p, {dh, u, du})) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const long long n8 = rows * (d_ff / 8);
    if (dtype == KLAB_BF16)
        geglu_bwd_kernel<__nv_bfloat16><<<geglu_grid(n8), GEGLU_THREADS, 0, st>>>(
            static_cast<const __nv_bfloat16*>(dh), static_cast<const __nv_bfloat16*>(u), static_cast<__nv_bfloat16*>(du), n8, d_ff / 8,
            seed, seed_ptr, p);
    else
        geglu_bwd_kernel<float><<<geglu_grid(n8), GEGLU_THREADS, 0, st>>>(static_cast<const float*>(dh), static_cast<const float*>(u),
                                                                          static_cast<float*>(du), n8, d_ff / 8, seed, seed_ptr, p);
    KLAB_LAUNCH_CHECK();
    count_launch();
    return KLAB_OK;
}

}  // extern "C"
