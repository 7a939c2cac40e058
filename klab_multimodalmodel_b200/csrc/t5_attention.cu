// K9 (generic path): T5 attention forward / backward, CUDA-core fp32 arithmetic, whole K/V of one (batch, head)
// resident in shared memory.  Follows T5Attention.forward, HF/models/t5/modeling_t5.py:253-344:
//   scores = q k^T (NO 1/sqrt(d) scale, :308) + bias[bucket(j - i)] (:236-251, table of block 0 shared by all
//   blocks, :758) [+ causal mask, :704]; softmax in fp32 (:331); dropout on the probabilities (:332); out = P v.
// q/k/v/o are read and written in the [B*L, H*d_kv] layout the projection GEMMs produce (no transposes).
// This kernel is exact-fp32 and serves the strict parity path for every shape; the bf16 hot path for
// d_kv = 64 is the tcgen05 kernel in t5_attention_tc.cu.
#include <cstdlib>

#include "common.cuh"

namespace klab {
void count_launch(int n = 1);
namespace {

constexpr int RPC = 16;     // rows per CTA
constexpr int NW = 4;       // warps per CTA

struct AttnArgs {
    const void *q, *k, *v, *o, *dout;
    void *out, *dq, *dk, *dv;
    long long ldq, ldk, ldv, ldo;      // ldo also used for dout / dq (ldq), dk (ldk), dv (ldv)
    int B, H, Lq, Lk, dk_;
    const float* bias_table;   // [num_buckets, H] or null
    const int* rel_bucket;     // bucket of relative position r = j - (i + q_offset); index r + rel_zero
    int rel_zero;
    int num_buckets;
    int causal;
    int q_offset;
    float* lse;                // [B, H, Lq]
    float* dvec;               // [B, H, Lq]  D_i = dO_i . O_i
    float* dbias_partial;      // [B*H*chunks, num_buckets]
    float dropout_p;
    unsigned long long seed;
    const unsigned long long* seed_ptr;
};

__device__ __forceinline__ float drop_mult(const AttnArgs& a, const DropKey& key, int bh, int i, int j) {
    if (!key.on) return 1.0f;
    const uint64_t idx = (static_cast<uint64_t>(bh) * a.Lq + i) * a.Lk + j;
    return dropout_mult(key, idx);
}

template <typename T>
__global__ void __launch_bounds__(NW * 32) t5_attn_fwd_kernel(AttnArgs a) {
    extern __shared__ float sm[];
    if (a.seed_ptr) a.seed += *a.seed_ptr;
    const int dk = a.dk_, Lk = a.Lk, Lq = a.Lq, dp = dk + 1;
    float* Ks = sm;
    float* Vs = Ks + Lk * dp;
    float* brel = Vs + Lk * dp;                 // [Lq + Lk]
    float* pbuf = brel + (Lq + Lk);             // [NW][Lk]
    float* qbuf = pbuf + NW * Lk;               // [NW][dk]
    const int bh = blockIdx.x, b = bh / a.H, h = bh % a.H;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const T* kp = reinterpret_cast<const T*>(a.k) + static_cast<long long>(b) * Lk * a.ldk + h * dk;
    const T* vp = reinterpret_cast<const T*>(a.v) + static_cast<long long>(b) * Lk * a.ldv + h * dk;
    for (int idx = threadIdx.x; idx < Lk * dk; idx += blockDim.x) {
        const int j = idx / dk, c = idx % dk;
        Ks[j * dp + c] = to_f32(kp[j * a.ldk + c]);
        Vs[j * dp + c] = to_f32(vp[j * a.ldv + c]);
    }
    if (a.bias_table)
        for (int r = threadIdx.x; r < Lq + Lk - 1; r += blockDim.x) {
            // r encodes (j - i) + (Lq - 1)
            const int rel = r - (Lq - 1) - a.q_offset;
            brel[r] = a.bias_table[a.rel_bucket[rel + a.rel_zero] * a.H + h];
        }
    __syncthreads();
    const DropKey dkey = make_drop_key(a.seed, a.dropout_p);
    float* pw = pbuf + warp * Lk;
    float* qw = qbuf + warp * dk;
    const int i_end = min(Lq, (static_cast<int>(blockIdx.y) + 1) * RPC);
    for (int i = blockIdx.y * RPC + warp; i < i_end; i += NW) {
        const T* qp = reinterpret_cast<const T*>(a.q) + (static_cast<long long>(b) * Lq + i) * a.ldq + h * dk;
        for (int c = lane; c < dk; c += 32) qw[c] = to_f32(qp[c]);
        __syncwarp();
        const int jmax = a.causal ? min(Lk, i + a.q_offset + 1) : Lk;     // keys [0, jmax) are visible
        float mx = -INFINITY;
        for (int j = lane; j < jmax; j += 32) {
            float s = 0.0f;
            const float* kr = Ks + j * dp;
#pragma unroll 8
            for (int c = 0; c < dk; ++c) s = fmaf(qw[c], kr[c], s);
            if (a.bias_table) s += brel[j - i + Lq - 1];
            pw[j] = s;
            mx = fmaxf(mx, s);
        }
        mx = warp_max(mx);
        float sum = 0.0f;
        for (int j = lane; j < jmax; j += 32) {
            const float e = __expf(pw[j] - mx);
            pw[j] = e;
            sum += e;
        }
        sum = warp_sum(sum);
        const float inv = 1.0f / sum;
        for (int j = lane; j < jmax; j += 32) pw[j] = pw[j] * inv * drop_mult(a, dkey, bh, i, j);
        __syncwarp();
        if (lane == 0) a.lse[(static_cast<long long>(bh)) * Lq + i] = mx + __logf(sum);
        T* op = reinterpret_cast<T*>(a.out) + (static_cast<long long>(b) * Lq + i) * a.ldo + h * dk;
        for (int c = lane; c < dk; c += 32) {
            float acc = 0.0f;
            for (int j = 0; j < jmax; ++j) acc = fmaf(pw[j], Vs[j * dp + c], acc);
            op[c] = from_f32<T>(acc);
        }
        __syncwarp();
    }
}

// Pass A of the backward: per query row -> dq, D_i, and the per-bucket bias gradient partials.
template <typename T>
__global__ void __launch_bounds__(NW * 32) t5_attn_bwd_dq_kernel(AttnArgs a) {
    extern __shared__ float sm[];
    if (a.seed_ptr) a.seed += *a.seed_ptr;
    const int dk = a.dk_, Lk = a.Lk, Lq = a.Lq, dp = dk + 1;
    float* Ks = sm;
    float* Vs = Ks + Lk * dp;
    float* brel = Vs + Lk * dp;                 // [Lq + Lk]
    int* relb = reinterpret_cast<int*>(brel + (Lq + Lk));   // [Lq + Lk]
    float* pbuf = reinterpret_cast<float*>(relb + (Lq + Lk));   // [NW][Lk]
    float* qbuf = pbuf + NW * Lk;               // [NW][dk]
    float* dobuf = qbuf + NW * dk;              // [NW][dk]
    float* s_dbias = dobuf + NW * dk;           // [num_buckets]
    const int bh = blockIdx.x, b = bh / a.H, h = bh % a.H;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const T* kp = reinterpret_cast<const T*>(a.k) + static_cast<long long>(b) * Lk * a.ldk + h * dk;
    const T* vp = reinterpret_cast<const T*>(a.v) + static_cast<long long>(b) * Lk * a.ldv + h * dk;
    for (int idx = threadIdx.x; idx < Lk * dk; idx += blockDim.x) {
        const int j = idx / dk, c = idx % dk;
        Ks[j * dp + c] = to_f32(kp[j * a.ldk + c]);
        Vs[j * dp + c] = to_f32(vp[j * a.ldv + c]);
    }
    if (a.bias_table) {
        for (int r = threadIdx.x; r < Lq + Lk - 1; r += blockDim.x) {
            const int rel = r - (Lq - 1) - a.q_offset;
            const int bk = a.rel_bucket[rel + a.rel_zero];
            relb[r] = bk;
            brel[r] = a.bias_table[bk * a.H + h];
        }
        for (int r = threadIdx.x; r < a.num_buckets; r += blockDim.x) s_dbias[r] = 0.0f;
    }
    __syncthreads();
    const DropKey dkey = make_drop_key(a.seed, a.dropout_p);
    float* pw = pbuf + warp * Lk;
    float* qw = qbuf + warp * dk;
    float* dow = dobuf + warp * dk;
    const int i_end = min(Lq, (static_cast<int>(blockIdx.y) + 1) * RPC);
    for (int i = blockIdx.y * RPC + warp; i < i_end; i += NW) {
        const long long row = static_cast<long long>(b) * Lq + i;
        const T* qp = reinterpret_cast<const T*>(a.q) + row * a.ldq + h * dk;
        const T* dop = reinterpret_cast<const T*>(a.dout) + row * a.ldo + h * dk;
        const T* op = reinterpret_cast<const T*>(a.o) + row * a.ldo + h * dk;
        float dsum = 0.0f;
        for (int c = lane; c < dk; c += 32) {
            qw[c] = to_f32(qp[c]);
            const float g = to_f32(dop[c]);
            dow[c] = g;
            dsum += g * to_f32(op[c]);
        }
        const float Di = warp_sum(dsum);
        __syncwarp();
        const float lse = a.lse[static_cast<long long>(bh) * Lq + i];
        const int jmax = a.causal ? min(Lk, i + a.q_offset + 1) : Lk;
        for (int j = lane; j < jmax; j += 32) {
            float s = 0.0f, dpv = 0.0f;
            const float* kr = Ks + j * dp;
            const float* vr = Vs + j * dp;
#pragma unroll 8
            for (int c = 0; c < dk; ++c) {
                s = fmaf(qw[c], kr[c], s);
                dpv = fmaf(dow[c], vr[c], dpv);
            }
            if (a.bias_table) s += brel[j - i + Lq - 1];
            const float p = __expf(s - lse);
            const float ds = p * (dpv * drop_mult(a, dkey, bh, i, j) - Di);
            pw[j] = ds;
            if (a.bias_table) atomicAdd(&s_dbias[relb[j - i + Lq - 1]], ds);
        }
        __syncwarp();
        if (lane == 0) a.dvec[static_cast<long long>(bh) * Lq + i] = Di;
        T* dqp = reinterpret_cast<T*>(a.dq) + row * a.ldq + h * dk;
        for (int c = lane; c < dk; c += 32) {
            float acc = 0.0f;
            for (int j = 0; j < jmax; ++j) acc = fmaf(pw[j], Ks[j * dp + c], acc);
            dqp[c] = from_f32<T>(acc);
        }
        __syncwarp();
    }
    if (a.bias_table) {
        __syncthreads();
        float* part = a.dbias_partial + (static_cast<long long>(bh) * gridDim.y + blockIdx.y) * a.num_buckets;
        for (int r = threadIdx.x; r < a.num_buckets; r += blockDim.x) part[r] = s_dbias[r];
    }
}

// Pass B of the backward: per key row -> dk, dv (probabilities recomputed from lse).
template <typename T>
__global__ void __launch_bounds__(NW * 32) t5_attn_bwd_dkv_kernel(AttnArgs a) {
    extern __shared__ float sm[];
    if (a.seed_ptr) a.seed += *a.seed_ptr;
    const int dk = a.dk_, Lk = a.Lk, Lq = a.Lq, dp = dk + 1;
    float* Qs = sm;
    float* dOs = Qs + Lq * dp;
    float* lse_s = dOs + Lq * dp;               // [Lq]
    float* d_s = lse_s + Lq;                    // [Lq]
    float* brel = d_s + Lq;                     // [Lq + Lk]
    float* pbuf = brel + (Lq + Lk);             // [NW][Lq]
    float* dsbuf = pbuf + NW * Lq;              // [NW][Lq]
    float* kbuf = dsbuf + NW * Lq;              // [NW][dk]
    float* vbuf = kbuf + NW * dk;               // [NW][dk]
    const int bh = blockIdx.x, b = bh / a.H, h = bh % a.H;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const T* qp = reinterpret_cast<const T*>(a.q) + static_cast<long long>(b) * Lq * a.ldq + h * dk;
    const T* dop = reinterpret_cast<const T*>(a.dout) + static_cast<long long>(b) * Lq * a.ldo + h * dk;
    for (int idx = threadIdx.x; idx < Lq * dk; idx += blockDim.x) {
        const int i = idx / dk, c = idx % dk;
        Qs[i * dp + c] = to_f32(qp[i * a.ldq + c]);
        dOs[i * dp + c] = to_f32(dop[i * a.ldo + c]);
    }
    for (int i = threadIdx.x; i < Lq; i += blockDim.x) {
        lse_s[i] = a.lse[static_cast<long long>(bh) * Lq + i];
        d_s[i] = a.dvec[static_cast<long long>(bh) * Lq + i];
    }
    if (a.bias_table)
        for (int r = threadIdx.x; r < Lq + Lk - 1; r += blockDim.x) {
            const int rel = r - (Lq - 1) - a.q_offset;
            brel[r] = a.bias_table[a.rel_bucket[rel + a.rel_zero] * a.H + h];
        }
    __syncthreads();
    const DropKey dkey = make_drop_key(a.seed, a.dropout_p);
    float* pw = pbuf + warp * Lq;
    float* dsw = dsbuf + warp * Lq;
    float* kw = kbuf + warp * dk;
    float* vw = vbuf + warp * dk;
    const int j_end = min(Lk, (static_cast<int>(blockIdx.y) + 1) * RPC);
    for (int j = blockIdx.y * RPC + warp; j < j_end; j += NW) {
        const long long krow = static_cast<long long>(b) * Lk + j;
        const T* kp = reinterpret_cast<const T*>(a.k) + krow * a.ldk + h * dk;
        const T* vp = reinterpret_cast<const T*>(a.v) + krow * a.ldv + h * dk;
        for (int c = lane; c < dk; c += 32) {
            kw[c] = to_f32(kp[c]);
            vw[c] = to_f32(vp[c]);
        }
        __syncwarp();
        const int imin = a.causal ? max(0, j - a.q_offset) : 0;      // queries [imin, Lq) see key j
        for (int i = imin + lane; i < Lq; i += 32) {
            float s = 0.0f, dpv = 0.0f;
            const float* qr = Qs + i * dp;
            const float* dor = dOs + i * dp;
#pragma unroll 8
            for (int c = 0; c < dk; ++c) {
                s = fmaf(qr[c], kw[c], s);
                dpv = fmaf(dor[c], vw[c], dpv);
            }
            if (a.bias_table) s += brel[j - i + Lq - 1];
            const float p = __expf(s - lse_s[i]);
            const float m = drop_mult(a, dkey, bh, i, j);
            pw[i] = p * m;
            dsw[i] = p * (dpv * m - d_s[i]);
        }
        __syncwarp();
        T* dkp = reinterpret_cast<T*>(a.dk) + krow * a.ldk + h * dk;
        T* dvp = reinterpret_cast<T*>(a.dv) + krow * a.ldv + h * dk;
        for (int c = lane; c < dk; c += 32) {
            float accv = 0.0f, acck = 0.0f;
            for (int i = imin; i < Lq; ++i) {
                accv = fmaf(pw[i], dOs[i * dp + c], accv);
                acck = fmaf(dsw[i], Qs[i * dp + c], acck);
            }
            dkp[c] = from_f32<T>(acck);
            dvp[c] = from_f32<T>(accv);
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------------------------------
// Decode shape (K14, HF/generation/utils.py:2743-2800 + HF/models/t5/modeling_t5.py:281-305): ONE query row per (batch, head)
// against the cached keys / values.  The work is reading K and V once (cross-attention: B * Le * 2 * inner bf16 per block and
// token, the largest HBM stream of a decode step), so the kernel is a bandwidth kernel: one warp per (b, h), 16-byte loads,
// LPR = d_kv / 8 lanes cover one row and 32 / LPR rows are in flight per load instruction; online softmax over chunks of keys
// whose K and V rows are requested together; fp32 arithmetic throughout.  A 128-row tensor-core tile would be > 97 % padding here.
// ------------------------------------------------------------------------------------------------------------------
constexpr int DEC_WARPS = 4;

__device__ __forceinline__ void unpack8_bf16(uint4 raw, float* f) {
    const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&raw);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 t = __bfloat1622float2(h2[i]);
        f[2 * i] = t.x;
        f[2 * i + 1] = t.y;
    }
}

template <int LPR>
__global__ void __launch_bounds__(DEC_WARPS * 32) t5_attn_decode_kernel(AttnArgs a) {
    constexpr int RPI = 32 / LPR;                 // key rows covered by one load instruction of the warp
    constexpr int CH = 8;                         // load instructions per chunk: RPI * CH keys are in flight per warp (K and V together)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int bh = blockIdx.x * DEC_WARPS + warp;
    if (bh >= a.B * a.H) return;
    const int b = bh / a.H, h = bh - b * a.H;
    const int Lk = a.Lk, dk = a.dk_;
    const int sub = lane % LPR, grp = lane / LPR;             // this lane covers columns [8 sub, 8 sub + 8) of row (j0 + c RPI + grp)
    const __nv_bfloat16* qp = reinterpret_cast<const __nv_bfloat16*>(a.q) + static_cast<long long>(b) * a.ldq + h * dk + 8 * sub;
    const __nv_bfloat16* kp = reinterpret_cast<const __nv_bfloat16*>(a.k) + static_cast<long long>(b) * Lk * a.ldk + h * dk + 8 * sub;
    const __nv_bfloat16* vp = reinterpret_cast<const __nv_bfloat16*>(a.v) + static_cast<long long>(b) * Lk * a.ldv + h * dk + 8 * sub;
    float q[8];
    unpack8_bf16(*reinterpret_cast<const uint4*>(qp), q);
    const int jmax = a.causal ? min(Lk, a.q_offset + 1) : Lk;         // keys [0, jmax) are visible to the single query row
    // online softmax over chunks of RPI * CH keys: the K and V rows of a chunk are requested together (one latency per chunk)
    float m = -INFINITY, l = 0.0f;
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int j0 = 0; j0 < jmax; j0 += RPI * CH) {
        uint4 kraw[CH], vraw[CH];
#pragma unroll
        for (int c = 0; c < CH; ++c) {
            const int j = j0 + c * RPI + grp;
            if (j < jmax) {
                kraw[c] = __ldg(reinterpret_cast<const uint4*>(kp + static_cast<long long>(j) * a.ldk));
                vraw[c] = __ldg(reinterpret_cast<const uint4*>(vp + static_cast<long long>(j) * a.ldv));
            } else {
                kraw[c] = make_uint4(0, 0, 0, 0);
                vraw[c] = make_uint4(0, 0, 0, 0);
            }
        }
        float sc[CH];
        float cm = -INFINITY;
#pragma unroll
        for (int c = 0; c < CH; ++c) {
            const int j = j0 + c * RPI + grp;
            float kf[8];
            unpack8_bf16(kraw[c], kf);
            float t = 0.0f;
#pragma unroll
            for (int i = 0; i < 8; ++i) t = fmaf(q[i], kf[i], t);
#pragma unroll
            for (int o = LPR / 2; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
            if (j < jmax) {
                if (a.bias_table) t += __ldg(a.bias_table + __ldg(a.rel_bucket + (j - a.q_offset) + a.rel_zero) * a.H + h);
                cm = fmaxf(cm, t);
            } else {
                t = -INFINITY;
            }
            sc[c] = t;
        }
#pragma unroll
        for (int o = LPR; o < 32; o <<= 1) cm = fmaxf(cm, __shfl_xor_sync(0xffffffffu, cm, o));
        const float m_new = fmaxf(m, cm);                             // finite: every chunk holds at least one visible key
        const float corr = __expf(m - m_new);                        // first chunk: exp(-inf) = 0
        l *= corr;
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i] *= corr;
#pragma unroll
        for (int c = 0; c < CH; ++c) {
            const float p = __expf(sc[c] - m_new);                   // masked rows: exp(-inf) = 0
            l += p;
            float vf[8];
            unpack8_bf16(vraw[c], vf);
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[i] = fmaf(p, vf[i], acc[i]);
        }
        m = m_new;
    }
    // combine the row groups of the warp (lanes with the same `sub` hold partial sums over different keys)
#pragma unroll
    for (int o = LPR; o < 32; o <<= 1) {
        l += __shfl_xor_sync(0xffffffffu, l, o);
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], o);
    }
    if (lane == 0) a.lse[bh] = m + __logf(l);
    if (grp == 0) {
        const float inv = 1.0f / l;
        uint4 outv;
        __nv_bfloat162* h2 = reinterpret_cast<__nv_bfloat162*>(&outv);
#pragma unroll
        for (int i = 0; i < 4; ++i) h2[i] = __floats2bfloat162_rn(acc[2 * i] * inv, acc[2 * i + 1] * inv);
        __nv_bfloat16* op = reinterpret_cast<__nv_bfloat16*>(a.out) + static_cast<long long>(b) * a.ldo + h * dk + 8 * sub;
        *reinterpret_cast<uint4*>(op) = outv;
    }
}

bool decode_shape_supported(int dtype, int Lq, int Lk, int dk, long long ldq, long long ldk, long long ldv, long long ldo, const void* q,
                            const void* k, const void* v, const void* o, float dropout_p) {
    if (dtype != KLAB_BF16 || Lq != 1 || dropout_p > 0.0f || Lk > 8192) return false;
    if (dk != 32 && dk != 64 && dk != 128) return false;
    if ((ldq | ldk | ldv | ldo) & 7) return false;
    return ((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k) | reinterpret_cast<uintptr_t>(v) | reinterpret_cast<uintptr_t>(o)) & 15) == 0;
}

int launch_decode(cudaStream_t st, const AttnArgs& a) {
    const int grid = (a.B * a.H + DEC_WARPS - 1) / DEC_WARPS;
    if (a.dk_ == 64) t5_attn_decode_kernel<8><<<grid, DEC_WARPS * 32, 0, st>>>(a);
    else if (a.dk_ == 32) t5_attn_decode_kernel<4><<<grid, DEC_WARPS * 32, 0, st>>>(a);
    else t5_attn_decode_kernel<16><<<grid, DEC_WARPS * 32, 0, st>>>(a);
    KLAB_LAUNCH_CHECK();
    count_launch();
    return KLAB_OK;
}

// dtable[bucket, h] += sum over (b, chunk) of partial[(b*H + h)*chunks + chunk][bucket]
__global__ void t5_dbias_reduce_kernel(const float* __restrict__ part, int B, int H, int chunks, int nb, float* __restrict__ dtable) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= nb * H) return;
    const int bucket = idx / H, h = idx % H;
    float s = 0.0f;
    for (int b = 0; b < B; ++b)
        for (int c = 0; c < chunks; ++c) s += part[((static_cast<long long>(b) * H + h) * chunks + c) * nb + bucket];
    dtable[idx] += s;
}

size_t fwd_smem(int Lq, int Lk, int dk) { return sizeof(float) * (2ll * Lk * (dk + 1) + (Lq + Lk) + NW * Lk + NW * dk); }
size_t dq_smem(int Lq, int Lk, int dk, int nb) {
    return sizeof(float) * (2ll * Lk * (dk + 1) + 2ll * (Lq + Lk) + NW * Lk + 2 * NW * dk + nb);
}
size_t dkv_smem(int Lq, int Lk, int dk) {
    return sizeof(float) * (2ll * Lq * (dk + 1) + 2ll * Lq + (Lq + Lk) + 2ll * NW * Lq + 2 * NW * dk);
}

template <typename K>
int set_smem(K kern, size_t bytes) {
    KLAB_REQUIRE(bytes <= 227 * 1024, "t5_attention: sequence too long for the resident-K/V kernel (%zu bytes of shared memory)", bytes);
    KLAB_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes)));
    return KLAB_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// Beam-search decode attention (klab_t5_attention_decode_beam): one query row per hypothesis, the nb hypotheses of one sample
// in consecutive rows.  One CTA per (sample, head) with one warp per beam; keys are streamed in chunks of CK through shared
// memory (fp32), online softmax per warp, fp32 arithmetic throughout (expf / fmaf: the fp32 variant is the exact path).
//   self-attention (src != null): key position j of row r lives in cache row src[r, j] * Lk + j -- the ancestry table replaces
//     HF's per-step cache reorder (cache.reorder_cache) -- with the causal bound j <= q_offset and the T5 relative bias;
//   cross-attention (src == null): all kv_group rows of a sample read that sample's [Lk, .] K/V, so each chunk is fetched once
//     per CTA and consumed by every beam: the cross K/V stream of a step does not grow with the number of beams.
// ------------------------------------------------------------------------------------------------------------------
struct BeamAttnArgs {
    const void *q, *k, *v;
    void* out;
    long long ldq, ldk, ldv, ldo;
    int G, H, Lk, dk;                 // G = rows per CTA (beams of a sample)
    const int* src;                   // [rows, ld_src] or null
    long long ld_src;
    const float* bias_table;
    const int* rel_bucket;
    int rel_zero, q_offset;
};

__device__ __forceinline__ void load_vec_f32(const __nv_bfloat16* p, float* dst) {      // 8 elements, one 16-byte load
    float f[8];
    unpack8_bf16(__ldg(reinterpret_cast<const uint4*>(p)), f);
#pragma unroll
    for (int i = 0; i < 8; ++i) dst[i] = f[i];
}
__device__ __forceinline__ void load_vec_f32(const float* p, float* dst) { dst[0] = __ldg(p); }

template <typename T, bool SELF, int CK>
__global__ void t5_attn_decode_beam_kernel(BeamAttnArgs a) {
    extern __shared__ float sm[];
    const int dk = a.dk, dp = dk + 1, G = a.G;
    constexpr int VEC = sizeof(T) == 2 ? 8 : 1;               // elements per load
    const int regions = SELF ? G : 1;
    float* Ks = sm;                                           // [regions][CK][dp]
    float* Vs = Ks + regions * CK * dp;
    float* qs = Vs + regions * CK * dp;                       // [G][dk]
    const int grp = blockIdx.x, h = blockIdx.y;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = grp * G + warp;
    const T* qp = reinterpret_cast<const T*>(a.q) + static_cast<long long>(row) * a.ldq + h * dk;
    for (int c = lane; c < dk; c += 32) qs[warp * dk + c] = to_f32(qp[c]);
    const int jmax = SELF ? min(a.Lk, a.q_offset + 1) : a.Lk;
    const int nthr = blockDim.x;
    const int per_row = dk / VEC;
    float m = -INFINITY, l = 0.0f;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};                      // columns lane + 32 i (d_kv <= 128)
    const float* Kw = Ks + (SELF ? warp : 0) * CK * dp;
    const float* Vw = Vs + (SELF ? warp : 0) * CK * dp;
    for (int j0 = 0; j0 < jmax; j0 += CK) {
        __syncthreads();                                      // previous chunk consumed
        for (int e = threadIdx.x; e < regions * CK * per_row; e += nthr) {
            const int g = e / (CK * per_row), rem = e % (CK * per_row), jj = rem / per_row, c = (rem % per_row) * VEC;
            const int j = j0 + jj;
            if (j >= jmax) continue;
            long long krow;
            if (SELF) krow = static_cast<long long>(__ldg(a.src + static_cast<long long>(grp * G + g) * a.ld_src + j)) * a.Lk + j;
            else krow = static_cast<long long>(grp) * a.Lk + j;
            const T* kp = reinterpret_cast<const T*>(a.k) + krow * a.ldk + h * dk + c;
            const T* vp = reinterpret_cast<const T*>(a.v) + krow * a.ldv + h * dk + c;
            float* kd = Ks + (g * CK + jj) * dp + c;
            float* vd = Vs + (g * CK + jj) * dp + c;
            load_vec_f32(kp, kd);
            load_vec_f32(vp, vd);
        }
        __syncthreads();
        const int j = j0 + lane;
        float sc = -INFINITY;
        if (lane < CK && j < jmax) {
            const float* kr = Kw + lane * dp;
            const float* qw = qs + warp * dk;
            float t = 0.0f;
            for (int c = 0; c < dk; ++c) t = fmaf(qw[c], kr[c], t);
            if (SELF && a.bias_table) t += __ldg(a.bias_table + __ldg(a.rel_bucket + (j - a.q_offset) + a.rel_zero) * a.H + h);
            sc = t;
        }
        const float m_new = fmaxf(m, warp_max(sc));                // finite: every chunk holds a visible key
        const float corr = expf(m - m_new);
        const float p = expf(sc - m_new);                          // masked lanes: exp(-inf) = 0
        l = l * corr + warp_sum(p);
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[i] *= corr;
        const int nk = min(CK, jmax - j0);
        for (int jj = 0; jj < nk; ++jj) {
            const float pj = __shfl_sync(0xffffffffu, p, jj);
            const float* vr = Vw + jj * dp;
#pragma unroll
            for (int i = 0; i < 4; ++i)
                if (lane + 32 * i < dk) acc[i] = fmaf(pj, vr[lane + 32 * i], acc[i]);
        }
        m = m_new;
    }
    const float inv = 1.0f / l;
    T* op = reinterpret_cast<T*>(a.out) + static_cast<long long>(row) * a.ldo + h * dk;
#pragma unroll
    for (int i = 0; i < 4; ++i)
        if (lane + 32 * i < dk) op[lane + 32 * i] = from_f32<T>(acc[i] * inv);
}

template <typename T, bool SELF, int CK>
int launch_decode_beam(cudaStream_t st, const BeamAttnArgs& a, int groups) {
    const int regions = SELF ? a.G : 1;
    const size_t smem = sizeof(float) * (2ull * regions * CK * (a.dk + 1) + 1ull * a.G * a.dk);
    if (int rc = set_smem(t5_attn_decode_beam_kernel<T, SELF, CK>, smem)) return rc;
    t5_attn_decode_beam_kernel<T, SELF, CK><<<dim3(groups, a.H), a.G * 32, smem, st>>>(a);
    KLAB_LAUNCH_CHECK();
    count_launch();
    return KLAB_OK;
}

}  // namespace

// tensor-core path (t5_attention_tc.cu)
bool t5_attention_tc_supported(int dtype, int Lq, int Lk, int d_kv, long long ldq, long long ldk, long long ldv, long long ldo,
                               const void* q, const void* k, const void* v, const void* o);
int t5_attention_fwd_tc(cudaStream_t st, int B, int H, int Lq, int Lk, const void* q, long long ldq, const void* k, long long ldk,
                        const void* v, long long ldv, void* out, long long ldo, const float* bias_table, const int* rel_bucket,
                        int rel_zero, int num_buckets, int causal, int q_offset, float* lse, float dropout_p, unsigned long long seed,
                        const unsigned long long* seed_ptr);
int t5_attention_bwd_tc(cudaStream_t st, int B, int H, int Lq, int Lk, const void* q, long long ldq, const void* k, long long ldk,
                        const void* v, long long ldv, const void* out, const void* dout, long long ldo, void* dq, void* dk, void* dv,
                        const float* bias_table, const int* rel_bucket, int rel_zero, int num_buckets, int causal, int q_offset,
                        const float* lse, float* dbias_table, float dropout_p, unsigned long long seed,
                        const unsigned long long* seed_ptr, void* workspace);
}  // namespace klab

using namespace klab;

static bool force_generic_attention() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("KLAB_ATTENTION_GENERIC");
        v = (e && e[0] == '1') ? 1 : 0;
    }
    return v == 1;
}

extern "C" {

long long klab_t5_attention_bwd_workspace_bytes(int B, int H, int Lq, int num_buckets) {
    const long long chunks = (Lq + RPC - 1) / RPC;
    return static_cast<long long>(sizeof(float)) * (1ll * B * H * Lq + 1ll * B * H * chunks * num_buckets);
}

int klab_t5_attention_fwd(void* stream, int dtype, int B, int H, int Lq, int Lk, int d_kv, const void* q, long long ldq,
                          const void* k, long long ldk, const void* v, long long ldv, void* out, long long ldo,
                          const float* bias_table, const int* rel_bucket, int rel_zero, int num_buckets, int causal,
                          int q_offset, float* lse, float dropout_p, unsigned long long seed,
                          const unsigned long long* seed_ptr) {
    if (int rc = klab_check_device()) return rc;
    KLAB_REQUIRE(B > 0 && H > 0 && Lq > 0 && Lk > 0 && d_kv > 0, "t5_attention_fwd: empty problem");
    if (decode_shape_supported(dtype, Lq, Lk, d_kv, ldq, ldk, ldv, ldo, q, k, v, out, dropout_p)) {      // Lq = 1: bandwidth kernel
        AttnArgs a{};
        a.q = q; a.k = k; a.v = v; a.out = out;
        a.ldq = ldq; a.ldk = ldk; a.ldv = ldv; a.ldo = ldo;
        a.B = B; a.H = H; a.Lq = Lq; a.Lk = Lk; a.dk_ = d_kv;
        a.bias_table = bias_table; a.rel_bucket = rel_bucket; a.rel_zero = rel_zero; a.num_buckets = num_buckets;
        a.causal = causal; a.q_offset = q_offset; a.lse = lse;
        return launch_decode(static_cast<cudaStream_t>(stream), a);
    }
    if (!force_generic_attention() && t5_attention_tc_supported(dtype, Lq, Lk, d_kv, ldq, ldk, ldv, ldo, q, k, v, out))
        return t5_attention_fwd_tc(static_cast<cudaStream_t>(stream), B, H, Lq, Lk, q, ldq, k, ldk, v, ldv, out, ldo, bias_table,
                                   rel_bucket, rel_zero, num_buckets, causal, q_offset, lse, dropout_p, seed, seed_ptr);
    AttnArgs a{};
    a.q = q; a.k = k; a.v = v; a.out = out;
    a.ldq = ldq; a.ldk = ldk; a.ldv = ldv; a.ldo = ldo;
    a.B = B; a.H = H; a.Lq = Lq; a.Lk = Lk; a.dk_ = d_kv;
    a.bias_table = bias_table; a.rel_bucket = rel_bucket; a.rel_zero = rel_zero; a.num_buckets = num_buckets;
    a.causal = causal; a.q_offset = q_offset; a.lse = lse; a.dropout_p = dropout_p; a.seed = seed; a.seed_ptr = seed_ptr;
    const size_t smem = fwd_smem(Lq, Lk, d_kv);
    const dim3 grid(B * H, (Lq + RPC - 1) / RPC);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (dtype == KLAB_BF16) {
        if (int rc = set_smem(t5_attn_fwd_kernel<__nv_bfloat16>, smem)) return rc;
        t5_attn_fwd_kernel<__nv_bfloat16><<<grid, NW * 32, smem, st>>>(a);
    } else {
        if (int rc = set_smem(t5_attn_fwd_kernel<float>, smem)) return rc;
        t5_attn_fwd_kernel<float><<<grid, NW * 32, smem, st>>>(a);
    }
    KLAB_LAUNCH_CHECK();
    count_launch();
    return KLAB_OK;
}

int klab_t5_attention_decode_beam(void* stream, int dtype, int rows, int H, int Lk, int d_kv, const void* q, long long ldq,
                                  const void* k, long long ldk, const void* v, long long ldv, void* out, long long ldo,
                                  int kv_group, const int* src, long long ld_src, const float* bias_table, const int* rel_bucket,
                                  int rel_zero, int q_offset) {
    if (int rc = klab_check_device()) return rc;
    KLAB_REQUIRE(rows > 0 && H > 0 && Lk > 0 && d_kv > 0 && d_kv <= 128 && kv_group >= 1 && kv_group <= 32 && rows % kv_group == 0,
                 "t5_attention_decode_beam: bad shape rows=%d H=%d Lk=%d d_kv=%d kv_group=%d", rows, H, Lk, d_kv, kv_group);
    KLAB_REQUIRE(!src || (q_offset >= 0 && q_offset < Lk && ld_src > q_offset), "t5_attention_decode_beam: q_offset %d outside the cache",
                 q_offset);
    if (dtype == KLAB_BF16)
        KLAB_REQUIRE(d_kv % 8 == 0 && ((ldq | ldk | ldv) & 7) == 0 &&
                     ((reinterpret_cast<uintptr_t>(k) | reinterpret_cast<uintptr_t>(v)) & 15) == 0,
                     "t5_attention_decode_beam: bf16 K/V need d_kv and row strides multiple of 8 and 16-byte aligned bases");
    BeamAttnArgs a{};
    a.q = q; a.k = k; a.v = v; a.out = out;
    a.ldq = ldq; a.ldk = ldk; a.ldv = ldv; a.ldo = ldo;
    a.G = kv_group; a.H = H; a.Lk = Lk; a.dk = d_kv;
    a.src = src; a.ld_src = ld_src; a.bias_table = bias_table; a.rel_bucket = rel_bucket; a.rel_zero = rel_zero; a.q_offset = q_offset;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int groups = rows / kv_group;
    if (dtype == KLAB_BF16)
        return src ? launch_decode_beam<__nv_bfloat16, true, 16>(st, a, groups) : launch_decode_beam<__nv_bfloat16, false, 32>(st, a, groups);
    return src ? launch_decode_beam<float, true, 16>(st, a, groups) : launch_decode_beam<float, false, 32>(st, a, groups);
}

int klab_t5_attention_bwd(void* stream, int dtype, int B, int H, int Lq, int Lk, int d_kv, const void* q, long long ldq,
                          const void* k, long long ldk, const void* v, long long ldv, const void* out, const void* dout,
                          long long ldo, void* dq, void* dk, void* dv, const float* bias_table, const int* rel_bucket,
                          int rel_zero, int num_buckets, int causal, int q_offset, const float* lse, float* dbias_table,
                          float dropout_p, unsigned long long seed, const unsigned long long* seed_ptr, void* workspace) {
    if (int rc = klab_check_device()) return rc;
    KLAB_REQUIRE(B > 0 && H > 0 && Lq > 0 && Lk > 0 && d_kv > 0, "t5_attention_bwd: empty problem");
    if (!force_generic_attention() && t5_attention_tc_supported(dtype, Lq, Lk, d_kv, ldq, ldk, ldv, ldo, q, k, v, out) &&
        (reinterpret_cast<uintptr_t>(dout) & 15) == 0)
        return t5_attention_bwd_tc(static_cast<cudaStream_t>(stream), B, H, Lq, Lk, q, ldq, k, ldk, v, ldv, out, dout, ldo, dq, dk, dv,
                                   bias_table, rel_bucket, rel_zero, num_buckets, causal, q_offset, lse, dbias_table, dropout_p, seed,
                                   seed_ptr, workspace);
    AttnArgs a{};
    a.q = q; a.k = k; a.v = v; a.o = out; a.dout = dout; a.dq = dq; a.dk = dk; a.dv = dv;
    a.ldq = ldq; a.ldk = ldk; a.ldv = ldv; a.ldo = ldo;
    a.B = B; a.H = H; a.Lq = Lq; a.Lk = Lk; a.dk_ = d_kv;
    a.bias_table = bias_table; a.rel_bucket = rel_bucket; a.rel_zero = rel_zero; a.num_buckets = num_buckets;
    a.causal = causal; a.q_offset = q_offset; a.lse = const_cast<float*>(lse); a.dropout_p = dropout_p; a.seed = seed; a.seed_ptr = seed_ptr;
    const int chunks = (Lq + RPC - 1) / RPC;
    a.dvec = static_cast<float*>(workspace);
    a.dbias_partial = a.dvec + 1ll * B * H * Lq;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t s1 = dq_smem(Lq, Lk, d_kv, num_buckets), s2 = dkv_smem(Lq, Lk, d_kv);
    const dim3 g1(B * H, chunks), g2(B * H, (Lk + RPC - 1) / RPC);
    if (dtype == KLAB_BF16) {
        if (int rc = set_smem(t5_attn_bwd_dq_kernel<__nv_bfloat16>, s1)) return rc;
        if (int rc = set_smem(t5_attn_bwd_dkv_kernel<__nv_bfloat16>, s2)) return rc;
        t5_attn_bwd_dq_kernel<__nv_bfloat16><<<g1, NW * 32, s1, st>>>(a);
        KLAB_LAUNCH_CHECK();
        t5_attn_bwd_dkv_kernel<__nv_bfloat16><<<g2, NW * 32, s2, st>>>(a);
    } else {
        if (int rc = set_smem(t5_attn_bwd_dq_kernel<float>, s1)) return rc;
        if (int rc = set_smem(t5_attn_bwd_dkv_kernel<float>, s2)) return rc;
        t5_attn_bwd_dq_kernel<float><<<g1, NW * 32, s1, st>>>(a);
        KLAB_LAUNCH_CHECK();
        t5_attn_bwd_dkv_kernel<float><<<g2, NW * 32, s2, st>>>(a);
    }
    KLAB_LAUNCH_CHECK();
    count_launch(2);
    if (bias_table && dbias_table) {
        const int n = num_buckets * H;
        t5_dbias_reduce_kernel<<<(n + 127) / 128, 128, 0, st>>>(a.dbias_partial, B, H, chunks, num_buckets, dbias_table);
        KLAB_LAUNCH_CHECK();
        count_launch();
    }
    return KLAB_OK;
}

}  // extern "C"
