// Beam search on device state: GenerationMixin._beam_search of HF 5.5.0 (HF/generation/utils.py:3076-3386), steps b-g of one
// iteration, for T5's single EOS id (beams_to_keep K = 2 * num_beams).  The host loop (generation.py: beam_generate) runs
//   LM-head GEMM -> beam_topk_kernel (per row: log_softmax + running score, top K) -> beam_update_kernel (per sample: merge,
//   stopping criteria, next running beams, finished set, early-stop heuristic, ancestry table)
// inside one CUDA-graph region per position; nothing goes back to the host except a "done" flag read every few steps.
//
// Ties resolve to the lower flat index beam * V + token everywhere (oracle/t5_beam.py: _topk_desc states the same rule).
#include "common.cuh"

namespace klab {
void count_launch(int n = 1);
namespace {

constexpr int TOPK_THREADS = 256;
constexpr float NEG_BIG = -1.0e9f;            // HF's mask value (:3195, :3013, :3048-3051)

__device__ __forceinline__ bool better(float va, long long ia, float vb, long long ib) { return va > vb || (va == vb && ia < ib); }

// One CTA per row of the fp32 logits [rows, V].  A single pass keeps an online max / sum of exp and, per thread, the K largest
// raw logits (each thread visits its columns in increasing order, so an equal later logit never displaces an earlier one).
// The thread lists are merged in K rounds of a block-wide argmax.  Output per row: the K pairs (log_softmax + running score,
// token id) in descending order, the log-probability computed as (x - max) - log(sum exp(x - max)) like torch's log_softmax.
// Selecting by raw logit is selecting by log-probability + score except where the fp32 rounding of that sum makes two
// different logits equal; the update kernel re-sorts by (value, flat index), and rounding ties only arise between -1e9 scores,
// whose candidates never reach the top K of their sample while it is live (see beam_update_kernel).
template <int K>
__global__ void __launch_bounds__(TOPK_THREADS) beam_topk_kernel(const float* __restrict__ logits, long long ld, int V,
                                                                  const float* __restrict__ run_scores, float* __restrict__ cand_val,
                                                                  int* __restrict__ cand_tok) {
    __shared__ float s_v[TOPK_THREADS / 32];
    __shared__ int s_i[TOPK_THREADS / 32];
    __shared__ float s_m[TOPK_THREADS / 32], s_s[TOPK_THREADS / 32];
    const int row = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float* x = logits + static_cast<long long>(row) * ld;
    float v[K];
    int id[K];
#pragma unroll
    for (int i = 0; i < K; ++i) { v[i] = -INFINITY; id[i] = 0x7fffffff; }
    float m = -INFINITY, s = 0.0f;
    for (int j = tid; j < V; j += TOPK_THREADS) {
        const float xv = __ldg(x + j);
        if (xv > m) { s = s * expf(m - xv) + 1.0f; m = xv; }
        else if (xv != -INFINITY) s += expf(xv - m);
        if (xv > v[K - 1] || id[K - 1] == 0x7fffffff) {
            v[K - 1] = xv;
            id[K - 1] = j;
#pragma unroll
            for (int i = K - 1; i > 0; --i)
                if (v[i] > v[i - 1] || (id[i - 1] == 0x7fffffff && id[i] != 0x7fffffff)) {
                    const float tv = v[i]; v[i] = v[i - 1]; v[i - 1] = tv;
                    const int ti = id[i]; id[i] = id[i - 1]; id[i - 1] = ti;
                }
        }
    }
    // block-wide (max, sum exp)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float m2 = __shfl_xor_sync(0xffffffffu, m, o), s2 = __shfl_xor_sync(0xffffffffu, s, o);
        const float mn = fmaxf(m, m2);
        s = (mn == -INFINITY) ? 0.0f : s * expf(m - mn) + s2 * expf(m2 - mn);
        m = mn;
    }
    if (lane == 0) { s_m[warp] = m; s_s[warp] = s; }
    __syncthreads();
    float M = -INFINITY;
    for (int w = 0; w < TOPK_THREADS / 32; ++w) M = fmaxf(M, s_m[w]);
    float S = 0.0f;
    for (int w = 0; w < TOPK_THREADS / 32; ++w) S += (s_m[w] == -INFINITY) ? 0.0f : s_s[w] * expf(s_m[w] - M);
    const float ls = logf(S);
    const float score = run_scores[row];
    // K rounds of block argmax over the heads of the thread lists
    for (int k = 0; k < K; ++k) {
        float bv = v[0];
        int bi = id[0];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
        }
        if (lane == 0) { s_v[warp] = bv; s_i[warp] = bi; }
        __syncthreads();
        bv = s_v[0];
        bi = s_i[0];
        for (int w = 1; w < TOPK_THREADS / 32; ++w)
            if (better(s_v[w], s_i[w], bv, bi)) { bv = s_v[w]; bi = s_i[w]; }
        if (id[0] == bi) {                                  // the owner pops its head
#pragma unroll
            for (int i = 0; i < K - 1; ++i) { v[i] = v[i + 1]; id[i] = id[i + 1]; }
            v[K - 1] = -INFINITY;
            id[K - 1] = 0x7fffffff;
        }
        if (tid == 0) {
            cand_val[static_cast<long long>(row) * K + k] = ((bv - M) - ls) + score;
            cand_tok[static_cast<long long>(row) * K + k] = bi;
        }
        __syncthreads();
    }
}

struct BeamArgs {
    const float* cand_val;          // [B*nb, K]
    const int* cand_tok;            // [B*nb, K]
    float* run_scores;              // [B*nb]
    int* src;                       // [2][B*nb][ld]   ancestry table, buffer (t & 1) is read, ((t + 1) & 1) written
    long long* run_seq;             // [2][B*nb][ld]
    float* fin_scores;              // [B*nb]
    long long* fin_seq;             // [2][B*nb][ld]
    int* fin_flag;                  // [B*nb]  is_sent_finished
    int* fin_len;                   // [B*nb]  generated length of the finished hypothesis (count of its beam indices)
    int* unsat;                     // [B]     is_early_stop_heuristic_unsatisfied
    int* done;                      // [B]     the sample's finished set can no longer change
    long long* next_tok;            // [B*nb]  input token of the next step
    int nb, V, T, t, eos;
    long long ld;                   // row length of src / run_seq / fin_seq (>= T + 1)
    float length_penalty;
    int early_stopping;             // 0: False, 1: True, 2: "never"
};

// One warp per sample.  A sample whose heuristic flag dropped, or (early_stopping True) whose finished set is full, is frozen:
// HF masks every later candidate of such a sample with -1e9 (:3048-3051), so its finished set never changes again, and this
// kernel stops changing it.  Its rows keep decoding (they are part of the batch) but their ancestry stays valid: a frozen
// step copies the tables forward with every row its own parent.
__global__ void __launch_bounds__(32) beam_update_kernel(BeamArgs a) {
    constexpr int KMAX = 16, NBMAX = 8;
    __shared__ float s_top_v[KMAX];
    __shared__ int s_top_parent[KMAX], s_top_tok[KMAX], s_hit[KMAX];
    __shared__ int s_run_from[NBMAX], s_run_tok[NBMAX];
    __shared__ float s_run_score[NBMAX];
    __shared__ int s_fin_from[NBMAX];              // < nb: old finished slot; >= nb: candidate (from - nb)
    __shared__ float s_fin_score[NBMAX];
    __shared__ int s_fin_flag[NBMAX], s_fin_len[NBMAX];
    __shared__ int s_frozen;
    const int b = blockIdx.x, lane = threadIdx.x;
    const int nb = a.nb, K = 2 * nb, t = a.t;
    const long long ld = a.ld;
    const int r0 = b * nb;
    const int cur = t & 1, nxt = cur ^ 1;
    const long long buf = static_cast<long long>(gridDim.x) * nb * ld;
    const int* src_c = a.src + cur * buf;
    int* src_n = a.src + nxt * buf;
    const long long* seq_c = a.run_seq + cur * buf;
    long long* seq_n = a.run_seq + nxt * buf;
    const long long* fin_c = a.fin_seq + cur * buf;
    long long* fin_n = a.fin_seq + nxt * buf;

    if (a.done[b]) {
        for (long long e = lane; e < static_cast<long long>(nb) * ld; e += 32) {
            const long long r = r0 + e / ld, j = e % ld;
            src_n[r * ld + j] = (j == t + 1) ? static_cast<int>(r) : src_c[r * ld + j];
            seq_n[r * ld + j] = seq_c[r * ld + j];
            fin_n[r * ld + j] = fin_c[r * ld + j];
        }
        return;
    }
    // b) top K of the sample's nb * K candidates by (value desc, flat index asc)
    const int n_cand = nb * K;
    float cv[4];
    long long cf[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int c = lane + 32 * i;
        if (c < n_cand) {
            const int beam = c / K;
            cv[i] = a.cand_val[static_cast<long long>(r0) * K + c];
            cf[i] = static_cast<long long>(beam) * a.V + a.cand_tok[static_cast<long long>(r0) * K + c];
        } else {
            cv[i] = -INFINITY;
            cf[i] = 0x7fffffffffffffffll;
        }
    }
    for (int k = 0; k < K; ++k) {
        float bv = cv[0];
        long long bf = cf[0];
        int bslot = 0;
#pragma unroll
        for (int i = 1; i < 4; ++i)
            if (better(cv[i], cf[i], bv, bf)) { bv = cv[i]; bf = cf[i]; bslot = i; }
        float wv = bv;
        long long wf = bf;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, wv, o);
            const long long of = __shfl_xor_sync(0xffffffffu, wf, o);
            if (better(ov, of, wv, wf)) { wv = ov; wf = of; }
        }
        if (bf == wf) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
                if (i == bslot) { cv[i] = -INFINITY; cf[i] = 0x7fffffffffffffffll; }
        }
        if (lane == 0) {
            s_top_v[k] = wv;
            s_top_parent[k] = static_cast<int>(wf / a.V);
            s_top_tok[k] = static_cast<int>(wf % a.V);
        }
    }
    __syncwarp();
    if (lane == 0) {
        const int cur_len = t + 1;
        const int max_length = a.T + 1;
        float rv[KMAX], fv[KMAX];
        bool taken[KMAX];
        const float denom = static_cast<float>(pow(static_cast<double>(cur_len), static_cast<double>(a.length_penalty)));
        for (int k = 0; k < K; ++k) {
            const int hit = (s_top_tok[k] == a.eos) || (cur_len + 1 >= max_length);        // EosTokenCriteria, MaxLengthCriteria
            s_hit[k] = hit;
            rv[k] = hit ? s_top_v[k] + NEG_BIG : s_top_v[k];                                // :3013
            const bool just = hit && k < nb;                                                // :3044
            fv[k] = s_top_v[k] / denom;                                                     // :3046
            if (!just) fv[k] += NEG_BIG;                                                    // :3051 (the :3049-3050 masks
            taken[k] = false;                                                               //  only hit frozen samples)
        }
        // c) next running beams: top nb of rv (:3016-3020)
        for (int i = 0; i < nb; ++i) {
            int best = -1;
            for (int k = 0; k < K; ++k)
                if (!taken[k] && (best < 0 || rv[k] > rv[best])) best = k;
            taken[best] = true;
            s_run_from[i] = r0 + s_top_parent[best];
            s_run_tok[i] = s_top_tok[best];
            s_run_score[i] = rv[best];
        }
        // d) finished set: top nb of [old finished scores, fv] (:3053-3064)
        float ms[NBMAX + KMAX];
        bool mt[NBMAX + KMAX];
        for (int i = 0; i < nb; ++i) { ms[i] = a.fin_scores[r0 + i]; mt[i] = false; }
        for (int k = 0; k < K; ++k) { ms[nb + k] = fv[k]; mt[nb + k] = false; }
        for (int i = 0; i < nb; ++i) {
            int best = -1;
            for (int c = 0; c < nb + K; ++c)
                if (!mt[c] && (best < 0 || ms[c] > ms[best])) best = c;
            mt[best] = true;
            s_fin_from[i] = best;
            s_fin_score[i] = ms[best];
            if (best < nb) {
                s_fin_flag[i] = a.fin_flag[r0 + best];
                s_fin_len[i] = a.fin_len[r0 + best];
            } else {
                s_fin_flag[i] = s_hit[best - nb] && (best - nb) < nb;
                s_fin_len[i] = t + 1;
            }
        }
        // e) early-stop heuristic after cur_len += 1 (:2876-2915)
        const int best_len = (a.early_stopping == 2 && a.length_penalty > 0.0f) ? a.T : cur_len;
        const float best_possible =
            s_run_score[0] / static_cast<float>(pow(static_cast<double>(best_len), static_cast<double>(a.length_penalty)));
        float mn = s_fin_score[0];
        bool all_fin = true;
        for (int i = 0; i < nb; ++i) { mn = fminf(mn, s_fin_score[i]); all_fin = all_fin && s_fin_flag[i]; }
        bool improvable = false;
        for (int i = 0; i < nb; ++i) improvable = improvable || best_possible > (s_fin_flag[i] ? mn : NEG_BIG);
        const int unsat = a.unsat[b] && improvable;
        a.unsat[b] = unsat;
        s_frozen = !unsat || (a.early_stopping == 1 && all_fin);
    }
    __syncwarp();
    // f) tables: running sequences and ancestry follow the parents; the finished set is rewritten from its sources
    for (long long e = lane; e < static_cast<long long>(nb) * ld; e += 32) {
        const int i = static_cast<int>(e / ld);
        const long long j = e % ld;
        const long long r = r0 + i, p = s_run_from[i];
        src_n[r * ld + j] = (j == t + 1) ? static_cast<int>(r) : src_c[p * ld + j];
        seq_n[r * ld + j] = (j == t + 1) ? static_cast<long long>(s_run_tok[i]) : seq_c[p * ld + j];
        const int from = s_fin_from[i];
        long long fvv;
        if (from < nb) {
            fvv = fin_c[(r0 + from) * ld + j];
        } else {
            const int k = from - nb;
            fvv = (j == t + 1) ? static_cast<long long>(s_top_tok[k]) : seq_c[(r0 + s_top_parent[k]) * ld + j];
        }
        fin_n[r * ld + j] = fvv;
    }
    __syncwarp();
    if (lane < nb) {
        a.run_scores[r0 + lane] = s_run_score[lane];
        a.next_tok[r0 + lane] = s_run_tok[lane];
        a.fin_scores[r0 + lane] = s_fin_score[lane];
        a.fin_flag[r0 + lane] = s_fin_flag[lane];
        a.fin_len[r0 + lane] = s_fin_len[lane];
    }
    if (lane == 0) a.done[b] = s_frozen;
}

}  // namespace
}  // namespace klab

using namespace klab;

extern "C" {

int klab_beam_topk(void* stream, int rows, int V, int k, const float* logits, long long ld, const float* run_scores, float* cand_val,
                   int* cand_tok) {
    if (int rc = klab_check_device()) return rc;
    KLAB_REQUIRE(rows > 0 && V >= k && k >= 4 && k <= 16 && (k & 1) == 0, "beam_topk: need rows > 0, k = 2 * num_beams in 4..16, V >= k");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    switch (k) {
#define KLAB_TOPK_CASE(KK) \
        case KK: beam_topk_kernel<KK><<<rows, TOPK_THREADS, 0, st>>>(logits, ld, V, run_scores, cand_val, cand_tok); break;
        KLAB_TOPK_CASE(4) KLAB_TOPK_CASE(6) KLAB_TOPK_CASE(8) KLAB_TOPK_CASE(10) KLAB_TOPK_CASE(12) KLAB_TOPK_CASE(14)
        KLAB_TOPK_CASE(16)
#undef KLAB_TOPK_CASE
    }
    KLAB_LAUNCH_CHECK();
    count_launch();
    return KLAB_OK;
}

int klab_beam_update(void* stream, int B, int nb, int V, int T, int t, int eos_id, float length_penalty, int early_stopping,
                     const float* cand_val, const int* cand_tok, float* run_scores, int* src, long long* run_seq, long long ld,
                     float* fin_scores, long long* fin_seq, int* fin_flag, int* fin_len, int* unsat, int* done, long long* next_tok) {
    if (int rc = klab_check_device()) return rc;
    KLAB_REQUIRE(B > 0 && nb >= 2 && nb <= 8 && V >= 2 * nb && t >= 0 && t < T && ld >= T + 1 && early_stopping >= 0 &&
                 early_stopping <= 2, "beam_update: bad arguments (B=%d nb=%d V=%d T=%d t=%d ld=%lld)", B, nb, V, T, t, ld);
    BeamArgs a{cand_val, cand_tok, run_scores, src, run_seq, fin_scores, fin_seq, fin_flag, fin_len, unsat, done, next_tok,
               nb, V, T, t, eos_id, ld, length_penalty, early_stopping};
    beam_update_kernel<<<B, 32, 0, static_cast<cudaStream_t>(stream)>>>(a);
    KLAB_LAUNCH_CHECK();
    count_launch();
    return KLAB_OK;
}

}  // extern "C"
