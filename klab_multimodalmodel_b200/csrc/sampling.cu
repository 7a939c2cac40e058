// Multinomial sampling step: GenerationMixin._sample of HF 5.5.0 (HF/generation/utils.py:2658-2800) for one token, with the
// three warpers transformers applies when sampling (HF/generation/logits_process.py), in its order:
//   temperature  s = logits / temperature                                        (TemperatureLogitsWarper, :236)
//   top-k        keep s >= the k-th largest s (ties at the k-th value are kept)   (TopKLogitsWarper, :536)
//   top-p        keep token i iff the softmax mass of the top-k-kept tokens with a strictly greater score is < top_p, or s_i is
//                the maximum (TopPLogitsWarper, :469; it sorts ascending and drops cumulative mass <= 1 - top_p, which is the
//                same set on rows without ties at the boundary -- this rule keeps every tied token; top_p = 0 keeps the maximum
//                and its ties)
// and a reproducible draw in place of torch.multinomial: u = u(seed, row, t - 1) (splitmix64 of a Weyl counter, 24 bits, see
// sample_u24), and the token is the smallest vocabulary index i with sum_{j <= i, kept} w_j > u * Z, w_j = exp(s_j - max),
// Z = sum over the kept tokens (the last kept token if rounding leaves none).  oracle/t5_sample.py states the same definition.
//
// One CTA of 1024 threads per row; the row is read from HBM once into shared memory (4 V bytes, 128.5 KB for T5's 32128) and
// everything else runs on chip: the max, the top-k threshold by a 4-pass radix select on the order-preserving uint32 key of
// the score (256-bin count histograms), the top-p threshold by the same radix select with mass-weighted histograms, and a
// vocabulary-order prefix scan for the inverse CDF.  Masses are fixed point, w * 2^40 in uint64, so every sum is exact and the
// token does not depend on the order in which threads add (the draw is deterministic run to run, graphs on or off).
#include "common.cuh"

namespace klab {
void count_launch(int n = 1);
namespace {

constexpr int SAMPLE_THREADS = 1024;
constexpr int SAMPLE_WARPS = SAMPLE_THREADS / 32;
constexpr float W_SCALE = 1099511627776.0f;                 // 2^40: Z < 2^56 for any V that fits in shared memory
constexpr unsigned FULL = 0xffffffffu;

struct SampleArgs {
    const float* logits;
    long long ld;
    long long* ids;
    long long ld_ids;
    int* unfinished;
    const unsigned long long* seed;
    int V, t, pad_id, eos_id, top_k;
    float temperature, top_p;
};

__device__ __forceinline__ unsigned order_key(float f) {            // a < b  <=>  key(a) < key(b)  (no NaNs)
    const unsigned b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

__device__ __forceinline__ float key_value(unsigned k) { return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k); }

__device__ __forceinline__ unsigned long long weight(float s, float m) { return __float2ull_rn(expf(s - m) * W_SCALE); }

// u(seed, row, c) * 2^24: splitmix64 (Steele, Lea, Flood 2014) finaliser of seed + golden-gamma * (1 + row * 2^16 + c)
__device__ __forceinline__ unsigned sample_u24(unsigned long long seed, long long row, int c) {
    unsigned long long z = seed + 0x9E3779B97F4A7C15ull * (1ull + static_cast<unsigned long long>(row) * 65536ull + static_cast<unsigned long long>(c));
    z ^= z >> 30;
    z *= 0xBF58476D1CE4E5B9ull;
    z ^= z >> 27;
    z *= 0x94D049BB133111EBull;
    z ^= z >> 31;
    return static_cast<unsigned>(z >> 40);
}

__device__ __forceinline__ unsigned long long warp_sum(unsigned long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

struct SelectSmem {
    unsigned long long hist[256];
    unsigned long long above;
    unsigned bin;
};

// Radix select from the top over the scores s[i] >= lo, each weighing 1 (MASS false) or w_i (MASS true): returns the key of
// the element at which the running total, taken from the largest score down, first reaches `goal`.  Four passes of 8 bits;
// histogram adds are aggregated per warp over lanes with the same bin (__match_any_sync), integer, so order-independent.
template <bool MASS>
__device__ unsigned select_from_top(const float* s, int V, float lo, float m, double goal, SelectSmem& sm) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    unsigned prefix = 0, pmask = 0;
    unsigned long long above = 0;
    for (int shift = 24; shift >= 0; shift -= 8) {
        if (tid < 256) sm.hist[tid] = 0;
        __syncthreads();
        for (int base = 0; base < V; base += SAMPLE_THREADS) {          // whole warps iterate together (warp intrinsics below)
            const int i = base + tid;
            const float x = i < V ? s[i] : -INFINITY;
            const unsigned key = order_key(x);
            const bool ok = i < V && x >= lo && (key & pmask) == prefix;
            const unsigned bin = ok ? (key >> shift) & 255u : 0xffffffffu;
            const unsigned grp = __match_any_sync(FULL, bin);
            if (ok) {
                unsigned long long add;
                if (MASS) {
                    const unsigned long long w = weight(x, m);         // < 2^41: two 20-bit halves never overflow a 32-lane sum
                    const unsigned hi = __reduce_add_sync(grp, static_cast<unsigned>(w >> 20));
                    const unsigned lo20 = __reduce_add_sync(grp, static_cast<unsigned>(w & 0xfffffull));
                    add = (static_cast<unsigned long long>(hi) << 20) + lo20;
                } else {
                    add = __popc(grp);
                }
                if (lane == __ffs(grp) - 1) atomicAdd(&sm.hist[bin], add);
            }
        }
        __syncthreads();
        if (warp == 0) {                                               // lane l holds bins 255 - 8l .. 248 - 8l (descending)
            unsigned long long c[8], sum = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) { c[j] = sm.hist[255 - 8 * lane - j]; sum += c[j]; }
            unsigned long long inc = sum;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long v = __shfl_up_sync(FULL, inc, o);
                if (lane >= o) inc += v;
            }
            const unsigned hit = __ballot_sync(FULL, static_cast<double>(above + inc) >= goal);
            const int f = hit ? __ffs(hit) - 1 : 31;                   // none: goal above the total (cannot happen), lowest bin
            if (lane == f) {
                unsigned long long run = above + inc - sum;
                int b = 255 - 8 * lane - 7;
                unsigned long long ab = run + sum - c[7];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    if (static_cast<double>(run + c[j]) >= goal) { b = 255 - 8 * lane - j; ab = run; break; }
                    run += c[j];
                }
                sm.bin = static_cast<unsigned>(b);
                sm.above = ab;
            }
        }
        __syncthreads();
        prefix |= sm.bin << shift;
        pmask |= 0xffu << shift;
        above = sm.above;
    }
    return prefix;
}

__global__ void __launch_bounds__(SAMPLE_THREADS, 1) sample_step_kernel(SampleArgs a) {
    extern __shared__ float4 s_row4[];
    float* s = reinterpret_cast<float*>(s_row4);                       // the row's scores, V floats
    __shared__ SelectSmem sel;
    __shared__ unsigned long long s_wsum[SAMPLE_WARPS];
    __shared__ float s_wmax[SAMPLE_WARPS];
    __shared__ int s_wlast[SAMPLE_WARPS];
    __shared__ int s_tok;
    const int row = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int V = a.V;
    long long* out = a.ids + static_cast<long long>(row) * a.ld_ids + a.t;
    if (!a.unfinished[row]) {                                          // finished rows emit pad (HF :2791)
        if (tid == 0) *out = a.pad_id;
        return;
    }
    if (tid == 0) s_tok = -1;
    // 1. the row into shared memory (temperature applied), and its max
    const float* x = a.logits + static_cast<long long>(row) * a.ld;
    const bool temp = a.temperature != 1.0f;
    float m = -INFINITY;
    if ((V & 3) == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0) {
        const float4* x4 = reinterpret_cast<const float4*>(x);
#pragma unroll 4
        for (int j = tid; j < (V >> 2); j += SAMPLE_THREADS) {
            float4 q = __ldg(x4 + j);
            if (temp) { q.x /= a.temperature; q.y /= a.temperature; q.z /= a.temperature; q.w /= a.temperature; }
            s_row4[j] = q;
            m = fmaxf(m, fmaxf(fmaxf(q.x, q.y), fmaxf(q.z, q.w)));
        }
    } else {
        for (int j = tid; j < V; j += SAMPLE_THREADS) {
            float q = __ldg(x + j);
            if (temp) q /= a.temperature;
            s[j] = q;
            m = fmaxf(m, q);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(FULL, m, o));
    if (lane == 0) s_wmax[warp] = m;
    __syncthreads();
    m = s_wmax[0];
#pragma unroll 8
    for (int w = 1; w < SAMPLE_WARPS; ++w) m = fmaxf(m, s_wmax[w]);
    const float mz = (m == -INFINITY) ? 0.0f : m;                       // an all -inf row: every weight is 0
    // 2. thresholds: kept = s >= tau
    float tau = -INFINITY;
    if (a.top_k > 0 && a.top_k < V) tau = key_value(select_from_top<false>(s, V, -INFINITY, mz, static_cast<double>(a.top_k), sel));
    if (a.top_p < 1.0f) {
        if (a.top_p <= 0.0f) {
            tau = m;
        } else {
            unsigned long long z = 0;
            for (int i = tid; i < V; i += SAMPLE_THREADS) {
                const float v = s[i];
                if (v >= tau) z += weight(v, mz);
            }
            z = warp_sum(z);
            if (lane == 0) s_wsum[warp] = z;
            __syncthreads();
            z = warp_sum(s_wsum[lane]);
            __syncthreads();                                           // s_wsum is reused below
            tau = key_value(select_from_top<true>(s, V, tau, mz, static_cast<double>(a.top_p) * static_cast<double>(z), sel));
        }
    }
    // 3. inverse CDF in vocabulary order: warp w owns [w * cw, (w + 1) * cw), its lanes reading consecutive scores
    const int cw = ((V + SAMPLE_THREADS - 1) / SAMPLE_THREADS) * 32;
    const int lo = min(V, warp * cw), hi = min(V, lo + cw);
    unsigned long long wsum = 0;
    int last = -1;
    for (int i = lo + lane; i < hi; i += 32) {
        const float v = s[i];
        if (v >= tau) { wsum += weight(v, mz); last = i; }
    }
    wsum = warp_sum(wsum);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) last = max(last, __shfl_xor_sync(FULL, last, o));
    if (lane == 0) { s_wsum[warp] = wsum; s_wlast[warp] = last; }
    __syncthreads();
    const unsigned long long mine = s_wsum[lane];
    const unsigned long long Z = warp_sum(mine);
    const unsigned long long excl = warp_sum(lane < warp ? mine : 0ull);
    const double target = static_cast<double>(sample_u24(*a.seed, row, a.t - 1)) * 0x1p-24 * static_cast<double>(Z);
    if (static_cast<double>(excl + s_wsum[warp]) > target && !(static_cast<double>(excl) > target)) {
        unsigned long long run = excl;
        for (int base = lo; base < hi; base += 32) {
            const int i = base + lane;
            float v = -INFINITY;
            if (i < hi) v = s[i];
            unsigned long long w = (i < hi && v >= tau) ? weight(v, mz) : 0ull;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long y = __shfl_up_sync(FULL, w, o);
                if (lane >= o) w += y;
            }
            const unsigned hit = __ballot_sync(FULL, static_cast<double>(run + w) > target);
            if (hit) {
                if (lane == 0) s_tok = base + __ffs(hit) - 1;
                break;
            }
            run += __shfl_sync(FULL, w, 31);
        }
    }
    __syncthreads();
    if (tid == 0) {
        int tok = s_tok;
        if (tok < 0) {                                                 // rounding left no index: the last kept token
            for (int w = 0; w < SAMPLE_WARPS; ++w) tok = max(tok, s_wlast[w]);
        }
        *out = tok;
        if (tok == a.eos_id) a.unfinished[row] = 0;
    }
}

}  // namespace
}  // namespace klab

using namespace klab;

extern "C" {

int klab_sample_step(void* stream, int rows, int V, const float* logits, long long ld, long long* ids, long long ld_ids, int t,
                     int* unfinished, int pad_id, int eos_id, float temperature, int top_k, float top_p,
                     const unsigned long long* seed) {
    if (int rc = klab_check_device()) return rc;
    KLAB_REQUIRE(rows > 0 && V > 0 && ld >= V && t >= 1 && t <= 65536 && ld_ids > t,
                 "sample_step: bad shape rows=%d V=%d ld=%lld t=%d ld_ids=%lld", rows, V, ld, t, ld_ids);
    KLAB_REQUIRE(temperature > 0.0f && temperature < INFINITY && top_k >= 0 && top_p >= 0.0f && seed != nullptr,
                 "sample_step: bad options temperature=%g top_k=%d top_p=%g (seed %p)", temperature, top_k, top_p, (const void*)seed);
    int dev = 0, optin = 0;
    KLAB_CHECK_CUDA(cudaGetDevice(&dev));
    KLAB_CHECK_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    cudaFuncAttributes fa{};
    KLAB_CHECK_CUDA(cudaFuncGetAttributes(&fa, sample_step_kernel));
    const size_t smem = static_cast<size_t>(V) * sizeof(float);
    KLAB_REQUIRE(smem + fa.sharedSizeBytes <= static_cast<size_t>(optin),
                 "sample_step: V=%d does not fit in shared memory (%zu + %zu bytes > %d)", V, smem, (size_t)fa.sharedSizeBytes, optin);
    KLAB_CHECK_CUDA(cudaFuncSetAttribute(sample_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    SampleArgs a{logits, ld, ids, ld_ids, unfinished, seed, V, t, pad_id, eos_id, top_k, temperature, top_p};
    sample_step_kernel<<<rows, SAMPLE_THREADS, smem, static_cast<cudaStream_t>(stream)>>>(a);
    KLAB_LAUNCH_CHECK();
    count_launch();
    return KLAB_OK;
}

}  // extern "C"
