// Prompt scoring: per-token log-probabilities, top-1 id and top-1 log-probability from the f32 logits rows of a prompt chunk.
//
// One CTA per row streams the row once with an online (running max, sum of exponentials) reduction and a running top-1, then
// reduces its threads in a fixed tree: the same inputs always give bit-identical outputs (no atomics on values).
//   logprob[t]    = logit[t][target[t]] - logsumexp(logit[t][0 .. vocab))      (NaN when target[t] == -1)
//   topId[t]      = lowest index of the largest logit among rows < limit      (the greedy arg-max rule of dl_engine_set_vocab_limit)
//   topLogprob[t] = logit[t][topId[t]] - logsumexp(...)
// The normaliser spans every vocabulary row of the model, as `dllama perplexity` does; only the top-1 honours the limit.
//
// Tensor parallel: every rank holds a vocabulary slice. Each rank reduces its slice to a per-row record {max, sum of exponentials
// relative to that max, top-1 value, top-1 global index, target logit (meaningful on the owning rank)} and pushes it as
// kScoreWordsPerRow LL words into every rank's slot area (one multimem.st through the NVSwitch multicast mapping, or nRanks unicast
// stores). Each rank then reads the nRanks records of the row, resets the words, and combines them in rank order, so every rank ends
// with bit-identical results. The waits are bounded spins, as in the prefill all-reduce (moe_prefill.cu: arResidualKernel).
#include <cmath>

#include "kernels.h"

namespace dl {
namespace {

constexpr int kScoreThreads = 512;

struct Rec {
    float m, s;     // running max and sum of exp(x - m)
    float v;        // top-1 value (-inf: none yet)
    int i;          // top-1 index (global)
};

// (m, s) += (m2, s2); exp(-inf) == 0 covers the empty operands
__device__ __forceinline__ void mergeMs(float &m, float &s, float m2, float s2) {
    if (m2 > m) {
        s = s * __expf(m - m2) + s2;
        m = m2;
    } else if (m2 > -INFINITY) {
        s = s + s2 * __expf(m2 - m);
    }
}

__device__ __forceinline__ void mergeTop(float &v, int &i, float v2, int i2) {
    if (v2 > v || (v2 == v && i2 < i)) { v = v2; i = i2; }
}

__device__ __forceinline__ void visit(Rec &r, float x, uint32_t idx, uint32_t rowOffset, uint32_t limit) {
    if (x > r.m) {
        r.s = r.s * __expf(r.m - x) + 1.0f;
        r.m = x;
    } else {
        r.s += __expf(x - r.m);
    }
    if (rowOffset + idx < limit && x > r.v) { r.v = x; r.i = (int)(rowOffset + idx); }   // increasing idx per thread: lowest index wins
}

__global__ void __launch_bounds__(kScoreThreads) scoreRowsKernel(ScoreArgs a, bool vec) {
    pdlLaunchDependents();
    pdlWait();
    const uint32_t t = blockIdx.x;
    const float *row = a.logits + (size_t)t * a.ld;
    const uint32_t limit = a.limit ? a.limit : 0xFFFFFFFFu;
    Rec r{-INFINITY, 0.f, -INFINITY, 0x7FFFFFFF};
    uint32_t tail = 0;
    if (vec) {
        const uint32_t n4 = a.vocab / 4;
        const float4 *row4 = reinterpret_cast<const float4 *>(row);
        for (uint32_t k = threadIdx.x; k < n4; k += kScoreThreads) {
            const float4 q = __ldcs(row4 + k);   // read once: do not keep the logits in L2
            visit(r, q.x, 4 * k, a.rowOffset, limit);
            visit(r, q.y, 4 * k + 1, a.rowOffset, limit);
            visit(r, q.z, 4 * k + 2, a.rowOffset, limit);
            visit(r, q.w, 4 * k + 3, a.rowOffset, limit);
        }
        tail = n4 * 4;
    }
    for (uint32_t k = tail + threadIdx.x; k < a.vocab; k += kScoreThreads) visit(r, __ldcs(row + k), k, a.rowOffset, limit);

    // fixed-shape tree: lanes, then the warps in index order
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float m2 = __shfl_down_sync(0xffffffffu, r.m, o), s2 = __shfl_down_sync(0xffffffffu, r.s, o);
        const float v2 = __shfl_down_sync(0xffffffffu, r.v, o);
        const int i2 = __shfl_down_sync(0xffffffffu, r.i, o);
        mergeMs(r.m, r.s, m2, s2);
        mergeTop(r.v, r.i, v2, i2);
    }
    __shared__ Rec warpRec[kScoreThreads / kWarp];
    const int warp = threadIdx.x / kWarp, lane = threadIdx.x % kWarp;
    if (lane == 0) warpRec[warp] = r;
    __syncthreads();
    if (threadIdx.x != 0) return;
    for (int w = 1; w < kScoreThreads / kWarp; w++) {
        mergeMs(r.m, r.s, warpRec[w].m, warpRec[w].s);
        mergeTop(r.v, r.i, warpRec[w].v, warpRec[w].i);
    }
    const int target = a.targets[t];
    const bool ownsTarget = target >= 0 && (uint32_t)target >= a.rowOffset && (uint32_t)target < a.rowOffset + a.vocab;
    float tgt = ownsTarget ? row[target - a.rowOffset] : 0.f;

    const ArArgs &ar = a.ar;
    if (ar.nRanks > 1) {
        // record words: {max, 1}, {sum, 1}, {top value, top index + 1}, {target logit, 1}; the flag half is never zero
        const uint32_t payload[kScoreWordsPerRow] = {__float_as_uint(r.m), __float_as_uint(r.s), __float_as_uint(r.v), __float_as_uint(tgt)};
        const uint32_t flag[kScoreWordsPerRow] = {1u, 1u, (uint32_t)r.i + 1u, 1u};
        const size_t cell = (size_t)t * kScoreWordsPerRow;
        const size_t mineOff = (size_t)(ar.parity * ar.nRanks + ar.rank) * ar.slotStride + cell;
        for (uint32_t k = 0; k < kScoreWordsPerRow; k++) {
            if (ar.slotsMc) {
                const uint64_t word = (uint64_t)payload[k] | ((uint64_t)flag[k] << 32);
                asm volatile("multimem.st.relaxed.sys.global.b64 [%0], %1;" ::"l"(ar.slotsMc + mineOff + k), "l"(word) : "memory");
            } else {
                for (uint32_t p = 0; p < ar.nRanks; p++) stLL(ar.slots[(ar.rank + p) % ar.nRanks] + mineOff + k, payload[k], flag[k]);
            }
        }
        uint64_t *mine = ar.slots[ar.rank];
        const uint32_t owner = target >= 0 ? (uint32_t)target / a.vocab : 0u;
        for (uint32_t sr = 0; sr < ar.nRanks; sr++) {
            uint2 w[kScoreWordsPerRow];
            for (uint32_t k = 0; k < kScoreWordsPerRow; k++) {
                uint64_t *p = mine + (size_t)(ar.parity * ar.nRanks + sr) * ar.slotStride + cell + k;
                w[k] = ldLL(p);
                uint32_t spins = 0;
                while (w[k].y == 0u && ++spins < (1u << 28)) w[k] = ldLL(p);
                stLL(p, 0u, 0u);
            }
            const float m2 = __uint_as_float(w[0].x), s2 = __uint_as_float(w[1].x), v2 = __uint_as_float(w[2].x);
            const int i2 = (int)w[2].y - 1;
            if (sr == 0) { r.m = m2; r.s = s2; r.v = v2; r.i = i2; }
            else { mergeMs(r.m, r.s, m2, s2); mergeTop(r.v, r.i, v2, i2); }
            if (sr == owner) tgt = __uint_as_float(w[3].x);
        }
    }
    const float logZ = r.m + __logf(r.s);
    a.outLogprob[t] = target >= 0 ? tgt - logZ : __int_as_float(0x7fc00000);
    a.outTopId[t] = r.v > -INFINITY ? r.i : -1;
    a.outTopLogprob[t] = r.v - logZ;
}

}  // namespace

int launchScoreRows(const ScoreArgs &a, cudaStream_t stream, bool pdl) {
    if (a.T == 0 || a.vocab == 0) return -1;
    const bool vec = a.ld % 4 == 0 && ((uintptr_t)a.logits & 15u) == 0;
    DL_CUDA_CHECK(launchPdl(scoreRowsKernel, dim3(a.T), dim3(kScoreThreads), 0, stream, pdl, a, vec));
    return 0;
}

}  // namespace dl

// Single-rank scoring of T logits rows (row t at logits + t * ldLogits, vocab entries): see the top of this file. limit 0 = none.
DL_EXPORT int dl_score_rows(const float *logits, uint32_t T, uint32_t vocab, uint32_t ldLogits, const int *targets, uint32_t limit,
                            float *outLogprob, int *outTopId, float *outTopLogprob, cudaStream_t stream) {
    dl::ScoreArgs a{};
    a.logits = logits; a.T = T; a.vocab = vocab; a.ld = ldLogits; a.targets = targets; a.limit = limit;
    a.outLogprob = outLogprob; a.outTopId = outTopId; a.outTopLogprob = outTopLogprob;
    return dl::launchScoreRows(a, stream, false);
}
