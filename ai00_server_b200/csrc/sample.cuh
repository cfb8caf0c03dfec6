// GPU front half of token sampling: penalties + allowed-token mask + bias + softmax + top-k, per slot, on the logits the
// head projection left in HBM.  Only <= 128 (token id, probability) pairs per slot cross PCIe.
//
// Replaces, for samplers that need only the head of the sorted distribution (Nucleus with top_k <= 128, greedy), what the
// reference does per generated token per slot (SURVEY.md §8f-1):
//   crates/ai00-core/src/run.rs:664-697   output.to_vec() (num_vocab f32 = 256 KiB D2H), Sampler::transform (penalties,
//                                         sampler/nucleus.rs:61-67), Formatter::transform (BNF mask, sampler/bnf.rs:37-40),
//                                         bias add (run.rs:679-681), softmax round trip (2 x 256 KiB, run.rs:1164-1190)
//   crates/ai00-core/src/sampler/nucleus.rs:69-80   full-vocabulary radix sort, `.rev().take(top_k)`
// The random draw, top_p cut, temperature and the penalty update (nucleus.rs:81-123) stay on the host: they need the
// sampler's state and RNG and touch <= top_k numbers.
//
// Order of the candidates: adjusted logit descending, token id ascending on ties -- a strict total order, so results are
// reproducible.  (The reference sorts probabilities with an unstable radix sort: any order of equal probabilities is a
// valid outcome there; this is one of them, because the probability is a non-decreasing function of the logit.)
//
// Shape: the vocabulary row (65536 f32 = 256 KB, L2 resident) is cut into 2048-element segments.
//   kernel 1 (grid = segments x rows): load, apply the two sparse lists and the mask, segment max / sum-exp, bitonic sort in
//            shared memory, keep the segment's best 128;
//   kernel 2 (grid = rows): combine the segment statistics into the softmax denominator (fixed order), merge the 32 sorted
//            lists pairwise -- the 128 best of two descending lists are first(a[i], b[127-i]), a bitonic sequence that seven
//            compare-exchange stages sort -- five rounds, then probabilities of the survivors.
// Nothing here is bandwidth: 16 rows x 256 KB from L2; two short launches.
#pragma once
#include "common.cuh"

namespace b200 {

constexpr int TOPK_MAX = 128;
constexpr int TOPK_SEG = 2048;            // elements per segment
constexpr int TOPK_SEG_THREADS = 256;
constexpr int TOPK_MAX_SEGS = 32;         // => num_vocab <= 65536
constexpr int TOPK_MERGE_THREADS = 1024;

struct TopkParams {
    const float* keep;          // [S][V] last logits row of every slot
    int V, nseg;
    const int* slot;            // [nrows]
    const int* pen_off;         // [nrows + 1]
    const unsigned* pen_tok;    // logits[tok] -= val   (entries of one row have distinct tokens)
    const float* pen_val;
    const int* bias_off;        // [nrows + 1]
    const unsigned* bias_tok;   // logits[tok] += val   (distinct tokens within a row)
    const float* bias_val;
    const unsigned* allow;      // optional [nrows][ceil(V / 32)]: bit = 1 -> token allowed; disallowed -> -inf
    float* cand_x;              // [nrows][nseg][128]
    unsigned* cand_id;          // [nrows][nseg][128]
    float2* stats;              // [nrows][nseg] (max, sum exp(x - max))
    int top_k;
    unsigned* out_id;           // [nrows][top_k]
    float* out_p;               // [nrows][top_k]
};

// strict total order: larger logit first, then smaller id
__device__ __forceinline__ bool cand_before(const float xa, const unsigned ia, const float xb, const unsigned ib) {
    return xa > xb || (xa == xb && ia < ib);
}

__global__ void __launch_bounds__(TOPK_SEG_THREADS) topk_segment_kernel(const __grid_constant__ TopkParams p) {
    __shared__ float sx[TOPK_SEG];
    __shared__ unsigned sid[TOPK_SEG];
    __shared__ float red[32];
    const int seg = blockIdx.x, row = blockIdx.y, tid = threadIdx.x;
    const int seg0 = seg * TOPK_SEG;
    const float* src = p.keep + (size_t)p.slot[row] * p.V;
    const unsigned* allow = p.allow ? p.allow + (size_t)row * ((p.V + 31) / 32) : nullptr;
#pragma unroll
    for (int j = 0; j < TOPK_SEG / TOPK_SEG_THREADS; ++j) {
        const int li = tid + TOPK_SEG_THREADS * j, i = seg0 + li;
        sx[li] = (i < p.V) ? src[i] : -INFINITY;
        sid[li] = (i < p.V) ? (unsigned)i : 0xFFFFFFFFu;
    }
    __syncthreads();
    // Sampler::transform: penalties (distinct tokens: race free)
    for (int e = p.pen_off[row] + tid; e < p.pen_off[row + 1]; e += TOPK_SEG_THREADS) {
        const unsigned t = p.pen_tok[e];
        if (t >= (unsigned)seg0 && t < (unsigned)(seg0 + TOPK_SEG) && t < (unsigned)p.V) sx[t - seg0] -= p.pen_val[e];
    }
    __syncthreads();
    // Formatter::transform: tokens the grammar does not allow
    if (allow) {
#pragma unroll
        for (int j = 0; j < TOPK_SEG / TOPK_SEG_THREADS; ++j) {
            const int li = tid + TOPK_SEG_THREADS * j, i = seg0 + li;
            if (i < p.V && !((allow[i >> 5] >> (i & 31)) & 1u)) sx[li] = -INFINITY;
        }
        __syncthreads();
    }
    // bias
    for (int e = p.bias_off[row] + tid; e < p.bias_off[row + 1]; e += TOPK_SEG_THREADS) {
        const unsigned t = p.bias_tok[e];
        if (t >= (unsigned)seg0 && t < (unsigned)(seg0 + TOPK_SEG) && t < (unsigned)p.V) sx[t - seg0] += p.bias_val[e];
    }
    __syncthreads();
    // segment statistics of the softmax
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < TOPK_SEG / TOPK_SEG_THREADS; ++j) mx = fmaxf(mx, sx[tid + TOPK_SEG_THREADS * j]);
    mx = block_max_any(mx, red);
    float s = 0.f;
    if (mx > -INFINITY) {
#pragma unroll
        for (int j = 0; j < TOPK_SEG / TOPK_SEG_THREADS; ++j) s += expf(sx[tid + TOPK_SEG_THREADS * j] - mx);
    }
    s = block_sum_any(s, red);
    if (tid == 0) p.stats[(size_t)row * p.nseg + seg] = make_float2(mx, s);
    // bitonic sort, best first
    for (int k = 2; k <= TOPK_SEG; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            __syncthreads();
#pragma unroll
            for (int q = 0; q < TOPK_SEG / 2 / TOPK_SEG_THREADS; ++q) {
                const int t = tid + TOPK_SEG_THREADS * q;            // compare-exchange index 0 .. 1023
                const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1)); // lower element of the pair
                const int l = i | j;
                const bool up = (i & k) == 0;                         // this block sorts best-first
                const float xa = sx[i], xb = sx[l];
                const unsigned ia = sid[i], ib = sid[l];
                const bool a_first = cand_before(xa, ia, xb, ib);
                if (a_first != up) { sx[i] = xb; sx[l] = xa; sid[i] = ib; sid[l] = ia; }
            }
        }
    }
    __syncthreads();
    if (tid < TOPK_MAX) {
        const size_t o = ((size_t)row * p.nseg + seg) * TOPK_MAX + tid;
        p.cand_x[o] = sx[tid];
        p.cand_id[o] = sid[tid];
    }
}

__global__ void __launch_bounds__(TOPK_MERGE_THREADS) topk_merge_kernel(const __grid_constant__ TopkParams p) {
    __shared__ float sx[TOPK_MAX_SEGS * TOPK_MAX];
    __shared__ unsigned sid[TOPK_MAX_SEGS * TOPK_MAX];
    __shared__ float s_m, s_inv;
    const int row = blockIdx.x, tid = threadIdx.x;
    for (int i = tid; i < TOPK_MAX_SEGS * TOPK_MAX; i += TOPK_MERGE_THREADS) {
        const int sg = i / TOPK_MAX;
        const bool ok = sg < p.nseg;
        const size_t o = ((size_t)row * p.nseg + sg) * TOPK_MAX + (i % TOPK_MAX);
        sx[i] = ok ? p.cand_x[o] : -INFINITY;
        sid[i] = ok ? p.cand_id[o] : 0xFFFFFFFFu;
    }
    if (tid < 32) {
        // softmax denominator from the segment statistics, fixed order (lane = segment, xor tree)
        const float2 st = (tid < p.nseg) ? p.stats[(size_t)row * p.nseg + tid] : make_float2(-INFINITY, 0.f);
        const float M = warp_max(st.x);
        float sc = (st.x > -INFINITY) ? st.y * expf(st.x - M) : 0.f;
        sc = warp_sum(sc);
        if (tid == 0) { s_m = M; s_inv = 1.0f / sc; }
    }
    // five merge rounds: lists a = 2 p s, b = (2 p + 1) s -> a
    for (int s = 1; s < TOPK_MAX_SEGS; s <<= 1) {
        const int npair = TOPK_MAX_SEGS / (2 * s);
        __syncthreads();
        for (int t = tid; t < npair * TOPK_MAX; t += TOPK_MERGE_THREADS) {
            const int pr = t / TOPK_MAX, i = t % TOPK_MAX;
            const int a = (2 * pr) * s * TOPK_MAX + i, b = (2 * pr + 1) * s * TOPK_MAX + (TOPK_MAX - 1 - i);
            if (!cand_before(sx[a], sid[a], sx[b], sid[b])) { sx[a] = sx[b]; sid[a] = sid[b]; }
        }
        for (int j = TOPK_MAX / 2; j > 0; j >>= 1) {
            __syncthreads();
            for (int t = tid; t < npair * (TOPK_MAX / 2); t += TOPK_MERGE_THREADS) {
                const int pr = t / (TOPK_MAX / 2), u = t % (TOPK_MAX / 2);
                const int i = (2 * pr) * s * TOPK_MAX + (((u & ~(j - 1)) << 1) | (u & (j - 1)));
                const int l = i + j;
                const float xa = sx[i], xb = sx[l];
                const unsigned ia = sid[i], ib = sid[l];
                if (!cand_before(xa, ia, xb, ib)) { sx[i] = xb; sx[l] = xa; sid[i] = ib; sid[l] = ia; }
            }
        }
    }
    __syncthreads();
    if (tid < p.top_k) {
        // same expression as softmax_kernel (misc.cuh): exp(x - max) * (1 / sum)
        p.out_id[(size_t)row * p.top_k + tid] = sid[tid];
        p.out_p[(size_t)row * p.top_k + tid] = (sx[tid] > -INFINITY) ? expf(sx[tid] - s_m) * s_inv : 0.f;
    }
}

// ---------------------------------------------------------------------------------------
// Last logits row of every slot that produced one in this step -> keep[slot][V].  The rows of a step are overwritten by
// the next step, which may belong to other slots (the reference samples every slot in its own task while the infer loop
// goes on, run.rs:1230-1240), so the front half above reads from this per-slot copy.  Tensor parallel: rank 0 gathers the
// vocabulary shards of all ranks (rows complete after the step's last rendezvous).
// ---------------------------------------------------------------------------------------
struct KeepParams {
    const float* shard[8];      // [R][Vl] logits shard of every rank (peer mapped)
    int world, Vl, V;
    MetaView meta;
    float* keep;                // [S][V]
};
constexpr int KEEP_THREADS = 256;
constexpr int KEEP_CHUNKS = 8;

__global__ void __launch_bounds__(KEEP_THREADS) keep_rows_kernel(const __grid_constant__ KeepParams p) {
    pdl_launch_dependents();
    const int r = blockIdx.x;
    const int R = p.meta.R();
    const int t = (r < R) ? p.meta.out_tok()[r] : 0;
    const bool live = r < R && p.meta.tok_last()[t] != 0;
    const int slot = live ? p.meta.tok_slot()[t] : 0;
    pdl_wait();
    if (!live) return;
    float* dst = p.keep + (size_t)slot * p.V;
    const int n4 = p.Vl >> 2;       // Vl % 4 == 0 is checked by the host
    for (int q = 0; q < p.world; ++q) {
        const float4* src = reinterpret_cast<const float4*>(p.shard[q] + (size_t)r * p.Vl);
        float4* d4 = reinterpret_cast<float4*>(dst + (size_t)q * p.Vl);
        for (int i = blockIdx.y * KEEP_THREADS + threadIdx.x; i < n4; i += KEEP_CHUNKS * KEEP_THREADS) d4[i] = __ldcg(src + i);
    }
}

// ---------------------------------------------------------------------------------------
// Scoring given tokens (b200rwkv_infer_score): logp = x[t] - m - log sum exp(x - m) of one logits row at one target id, for
// a list of (source row, target, destination).  This is the reference's perplexity() (crates/ai00-core/src/run.rs:699-755),
// which copies every row to the host and normalises it there only to read back one number.
// One CTA per row: each thread keeps an online (max, sum exp) over its strided share of the row (L2 resident, read once),
// then warps and the block combine the pairs in a fixed order -- no float atomics, so the result is bit-reproducible.
// Sources: a row of this step's logits (tensor parallel: rank 0 reads the vocabulary shard of every rank, complete after the
// step's last rendezvous), or keep[slot] (already gathered) for the first token of a SCORE_KEPT entry.
// ---------------------------------------------------------------------------------------
struct ScoreItem {
    int src;                    // >= 0: output row of the step;  < 0: keep[-src - 1]
    unsigned target;            // token id whose log-probability is wanted
    int dst;                    // index into logp
    int pad;
};
struct ScoreParams {
    const float* shard[8];      // [R][Vl] logits shard of every rank (peer mapped)
    int world, Vl, V;
    const float* keep;          // [S][V]
    const ScoreItem* items;     // [gridDim.x]
    float* logp;
};
constexpr int SCORE_THREADS = 512;

__device__ __forceinline__ void lse_push(float& m, float& s, const float x) {
    if (x > m) { s = s * expf(m - x) + 1.f; m = x; }
    else s += expf(x - m);
}
__device__ __forceinline__ void lse_merge(float& m, float& s, const float m2, const float s2) {
    const float M = fmaxf(m, m2);
    if (M == -INFINITY) return;                      // both halves empty
    s = s * expf(m - M) + s2 * expf(m2 - M);         // commutative: both lanes of a butterfly agree bit for bit
    m = M;
}

__global__ void __launch_bounds__(SCORE_THREADS) score_rows_kernel(const __grid_constant__ ScoreParams p) {
    __shared__ float red_m[SCORE_THREADS / 32], red_s[SCORE_THREADS / 32];
    const ScoreItem it = p.items[blockIdx.x];
    const bool kept = it.src < 0;
    const int nsh = kept ? 1 : p.world, w = kept ? p.V : p.Vl;
    float m = -INFINITY, s = 0.f;
    for (int q = 0; q < nsh; ++q) {
        const float* row = kept ? p.keep + (size_t)(-it.src - 1) * p.V : p.shard[q] + (size_t)it.src * p.Vl;
        if ((w & 3) == 0) {
            const float4* r4 = reinterpret_cast<const float4*>(row);
            for (int i = threadIdx.x; i < (w >> 2); i += SCORE_THREADS) {
                const float4 v = __ldcg(r4 + i);
                lse_push(m, s, v.x); lse_push(m, s, v.y); lse_push(m, s, v.z); lse_push(m, s, v.w);
            }
        } else {
            for (int i = threadIdx.x; i < w; i += SCORE_THREADS) lse_push(m, s, __ldcg(row + i));
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) lse_merge(m, s, __shfl_xor_sync(0xffffffffu, m, o), __shfl_xor_sync(0xffffffffu, s, o));
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { red_m[warp] = m; red_s[warp] = s; }
    __syncthreads();
    if (warp != 0) return;
    m = lane < SCORE_THREADS / 32 ? red_m[lane] : -INFINITY;
    s = lane < SCORE_THREADS / 32 ? red_s[lane] : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) lse_merge(m, s, __shfl_xor_sync(0xffffffffu, m, o), __shfl_xor_sync(0xffffffffu, s, o));
    if (lane == 0) {
        const int tq = kept ? 0 : (int)(it.target / (unsigned)p.Vl);
        const float* row = kept ? p.keep + (size_t)(-it.src - 1) * p.V : p.shard[tq] + (size_t)it.src * p.Vl;
        const float xt = __ldcg(row + (kept ? it.target : it.target - (unsigned)tq * p.Vl));
        p.logp[it.dst] = (xt - m) - logf(s);
    }
}

}  // namespace b200
