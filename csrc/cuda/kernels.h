// Internal C++ interface between the kernel translation units and the engine.
#pragma once
#include "common.cuh"

namespace dl {

enum { PRO_RMSNORM_ = 0, PRO_PLAIN_ = 1 };
enum { EPI_STORE_ = 0, EPI_RESIDUAL_ = 1, EPI_SWIGLU_ = 2, EPI_ARGMAX_ = 3, EPI_MOE_DOWN_ = 4 };

// In-kernel one-shot all-reduce over NVLink peer memory (see the EPI_RESIDUAL epilogue of gemv_q40_tma.cu).
constexpr int kMaxRanks = 8;
extern uint32_t gHiddenAct;   // process-wide gate activation (0 = SiLU, 1 = GELU), set by dl_engine_create from the model header

struct ArArgs {
    uint32_t nRanks, rank, parity, maxCtas;
    uint32_t slotStride;          // words per (parity, source rank) slot = maxBatch * dim
    uint32_t dim;                 // words between tokens inside a slot
    uint64_t *slots[kMaxRanks];   // rank r's LL slot area, mapped into this process: [2][nRanks][slotStride] x (f32 payload, flag)
    uint64_t *cand[kMaxRanks];    // rank r's arg-max candidates: [nRanks] x (f32 value, index + 1)
    uint64_t *slotsMc;            // NVLS multicast mapping of the slot area (one multimem.st reaches every rank), or null
};

struct GemvArgs {
    const uint32_t *qs;
    const __half *scales;
    uint32_t d, n;
    const float *in;
    const float *normW;
    float eps;
    float *out;
    uint32_t inStride, outStride;
    uint32_t maxTileRows;
    const int *expertIdx;
    uint32_t slot, kActive;
    uint64_t expertQsStride, expertScaleStride;
    const float *expertWeight;
    // EPI_ARGMAX (TMA kernel, nb == 1): logits are stored and the greedy token is selected in the same launch
    float *argVal;            // [grid] per-CTA best value
    int *argIdx;              // [grid] per-CTA best index
    unsigned int *argCounter; // zero-initialised, self-resetting
    int *tokenOut, *posInOut, *history;
    uint32_t historyCap;
    uint32_t rowOffsetGlobal; // added to row indices (vocab slice offset under tensor parallelism)
    uint64_t *trace;          // optional 4-slot timeline record for this launch
    // Mixture-of-experts launches (moeCtasPerSlot > 0, nb == 1): CTA b works for routing slot b / moeCtasPerSlot on the row
    // tile b % moeCtasPerSlot of expert expertIdx[slot]; experts outside [moeFirstExpert, +moeNumLocal) are skipped (EP).
    uint32_t moeCtasPerSlot, moeFirstExpert, moeNumLocal;
    uint32_t inSlotStride, outSlotStride;   // floats between slots of the input (w2) / output (w13) buffers
    float *moeScratch;          // [kActive][d] weighted per-slot products (EPI_MOE_DOWN)
    unsigned int *moeCounters;  // [moeCtasPerSlot], zero-initialised, self-resetting
    ArArgs ar;                // ar.nRanks > 1: EPI_RESIDUAL sums the partial products of all ranks before the residual add
    uint32_t act;             // gate activation of EPI_SWIGLU (filled in by the launchers from gHiddenAct)
    uint32_t vocabLimit;      // EPI_ARGMAX: rows (global index) >= vocabLimit never win (model vocabulary padded beyond the tokenizer's); 0 = no limit
};
int gemvQ40(int pro, int epi, int nb, GemvArgs a, int numSms, cudaStream_t stream, bool pdl);      // per-thread loads (fallback)
int gemvQ40Tma(int pro, int epi, int nb, GemvArgs a, int numSms, cudaStream_t stream, bool pdl);   // TMA ring; returns 1 if shape unsupported
inline int gemvQ40Auto(int pro, int epi, int nb, const GemvArgs &a, int numSms, cudaStream_t stream, bool pdl) {
    const int r = gemvQ40Tma(pro, epi, nb, a, numSms, stream, pdl);
    return r == 1 ? gemvQ40(pro, epi, nb, a, numSms, stream, pdl) : r;
}

// f32 / f16 weight files (gemv_dense.cu): wtype 1 = f32, 2 = f16; a.qs is the row-major [d][n] matrix
int gemvDense(int wtype, int pro, int epi, int nb, GemvArgs a, int numSms, cudaStream_t stream, bool pdl);

struct RopeKvArgs {
    float *qkv;
    uint32_t qkvStride;
    const int *pos;
    const float *rope;
    const float *qNorm;
    const float *kNorm;
    float eps;
    uint32_t nHeads, nKvHeads, headDim, seqLen;
    __nv_bfloat16 *kCache;
    __nv_bfloat16 *vCache;
};
int launchRopeKv(const RopeKvArgs &a, int nb, cudaStream_t stream, bool pdl);

struct AttnArgs {
    const float *qkv;
    uint32_t qkvStride;
    const int *pos;
    const __nv_bfloat16 *kCache, *vCache;
    uint32_t nHeads, nKvHeads, headDim, seqLen, nSplits;
    float *partial;
    unsigned int *counters;
    float *out;
    uint32_t outStride;
    __nv_bfloat16 *outBf16;   // if set, the result is written here (bf16) instead of `out`
};
int launchAttnDecode(const AttnArgs &a, int nb, cudaStream_t stream, bool pdl);

// Prompt-chunk attention on tcgen05 (attn_prefill_tc.cu): T consecutive tokens at positions p0.., causal, GQA heads packed on MMA-M.
struct AttnPrefillArgs {
    const float *qkv;            // [T][qkvStride] f32, q rows already normalised + rotated; K/V of the chunk already in the cache
    uint32_t qkvStride;
    uint32_t T, p0;
    uint32_t nHeads, nKvHeads, headDim, seqLen;
    const __nv_bfloat16 *kCache, *vCache;   // [nKvHeads][seqLen][headDim]
    __nv_bfloat16 *out;          // [T][outStride], head h at columns h * headDim
    uint32_t outStride;
};
int launchAttnPrefillTc(const AttnPrefillArgs &a, cudaStream_t stream, bool pdl = false);   // 1: shape not covered

// Single-token decode attention with QK-norm + RoPE + KV-cache append fused in (no separate rope kernel).
struct AttnFusedArgs {
    const float *qkv;        // raw q|k|v row of the token (f32, straight from the QKV GEMV)
    const int *pos;
    const float *rope;       // [seqLen][hd/2][2]
    const float *qNorm, *kNorm;
    float eps;
    __nv_bfloat16 *kCache, *vCache;
    uint32_t nHeads, nKvHeads, headDim, seqLen, nSplits;
    float *partial;
    unsigned int *counters;
    float *out;
    uint64_t *trace;
};
int launchAttnFused(const AttnFusedArgs &a, cudaStream_t stream, bool pdl);

struct RouterArgs {
    const float *x;            // [nb][dim] residual stream
    const float *normW;        // [dim]
    const float *gate;         // [nExperts][dim] f32
    float eps;
    uint32_t dim, nExperts, k;
    float *logits;             // [nb][nExperts] scratch
    unsigned int *counter;     // [nb], zero-initialised, self-resetting
    int *expertIdx;            // [nb][k]
    float *expertWeight;       // [nb][k]
};
int launchMoeRouter(const RouterArgs &a, int nb, cudaStream_t stream, bool pdl);

// Token embedding table (f32 [vocab][dim]). Tensor parallel: sharded by vocabulary rows over the ranks' peer-mapped memory — rank r
// holds rows [r * rowsPerRank, (r + 1) * rowsPerRank) and every rank reads the row of the current token straight from its owner over
// NVLink (reference K1: the root embeds and broadcasts x, src/llm.cpp:248-256; here a 16 KB peer load replaces 2.1 GB x N of replicas).
struct EmbTable {
    const float *shard[kMaxRanks];   // shard[0] is the whole table when rowsPerRank == 0
    uint32_t rowsPerRank;
    __host__ __device__ const float *row(uint32_t tok, uint32_t dim) const {
        if (rowsPerRank == 0) return shard[0] + (size_t)tok * dim;
        const uint32_t r = tok / rowsPerRank;
        return shard[r] + (size_t)(tok - r * rowsPerRank) * dim;
    }
};
int launchEmbedding(const EmbTable &table, const int *tokens, float *x, uint32_t dim, uint32_t xStride, uint32_t vocab, int nb,
                    cudaStream_t stream);
int launchArgmaxAdvance(const float *logits, uint32_t vocab, int *tokenOut, int *pos, int *history, uint32_t historyCap,
                        cudaStream_t stream, bool pdl);   // single rank only: the index is local to `logits`

// Device-side temperature / top-p sampler and the logits gather that feeds it under tensor parallelism (sampler.cu)
int launchSample(const float *logits, float *probs, uint32_t n, float temperature, float topp, unsigned long long *rng, int *tokenOut, int *pos,
                 int *history, uint32_t historyCap, const unsigned int *gatherFlag, unsigned int *gatherEpoch, uint32_t nRanks,
                 cudaStream_t stream);
int launchLogitsGather(const float *local, uint32_t v0, uint32_t rank, uint32_t nRanks, float *gatherMc, float *const *gatherUcDev,
                       unsigned int *flagMc, unsigned int *const *flagUcDev, unsigned int *blockCounter, cudaStream_t stream);

// Persistent decode kernel (mega_decode.cu)
struct MegaLayer {
    const uint8_t *qkvQs, *qkvSc, *woQs, *woSc, *w13Qs, *w13Sc, *w2Qs, *w2Sc;
    const float *norm0, *norm1, *qNorm, *kNorm;
    __nv_bfloat16 *kCache, *vCache;
};

struct MegaPhase {   // host-computed geometry of one GEMV phase (QKV, WO, W1|W3, W2, logits)
    uint32_t d, n, nblk, nseg;
    uint32_t stageRows;            // rows per ring fill (multiple of 4)
    uint32_t pairsQ, pairsRem;     // row pairs per CTA: CTA b owns pairsQ + (b < pairsRem) pairs starting at b*pairsQ + min(b, pairsRem)
    uint32_t recipNseg, gInc, segInc, rotInc;   // step -> (row group, segment) bookkeeping without divisions
};

struct MegaArgs {
    const MegaLayer *layers;     // [nLayers] in global memory
    uint32_t nLayers, dim, nHeads, nKvHeads, headDim, ffDim, vocab, vocabFull, seqLen, nSplits;
    float eps;
    EmbTable embedding;
    const float *finalNorm, *rope;
    const uint8_t *wclsQs, *wclsSc;
    int *tokens, *pos, *history;
    float *logits;
    uint2 *xW2;                  // second residual buffer (barrier-free hand-off experiment, flags bit 0)
    uint32_t flags;
    uint2 *xW, *qkvW, *zW;       // phase-crossing vectors as LL words {f32, epoch} (engine-owned, see mega_decode.cu)
    float *hF;                   // SwiGLU vector: plain f32 behind a fenced barrier (too large to pay the 2x LL footprint)
    unsigned int *launchSeq;     // device-resident launch counter (epoch base)
    unsigned int *abortFlag;     // host-mapped: set by a wait loop that ran out of its spin budget
    unsigned long long *syncNs;  // device accumulator: ns CTA 0 spent waiting for peer ranks in the all-reduce epilogues (null: off)
    float *attnPartial;
    unsigned int *attnCounters;
    float *argVal;
    int *argIdx;
    unsigned int *argCounter;
    unsigned int *gridCounter;   // zeroed by a memset node before every launch
    uint32_t stageBytes, nStages, planeBlocks, partialFloats;   // shared-memory geometry (host computed)
    uint32_t maxInflight;        // producer pacing: bulk-copy fills outstanding per CTA (0 = the whole ring)
    MegaPhase ph[5];
    uint32_t rowOffsetGlobal;
    uint32_t greedyAdvance;      // 1: publish the arg-max token and advance the position on the device
    uint32_t act, vocabLimit;    // see GemvArgs
    uint64_t *trace;
    uint32_t traceCtas, traceStride;   // CTAs 0..traceCtas-1 record their phase stamps at trace[cta * traceStride + slot]
    ArArgs ar;
};

int launchMegaDecode(MegaArgs m, int numSms, cudaStream_t stream);

// tcgen05 prefill GEMM (gemm_q40_tc.cu)
enum { GEPI_STORE_F32_ = 0, GEPI_RESIDUAL_ = 1, GEPI_SWIGLU_BF16_ = 2, GEPI_STORE_BF16_ = 3 };
int gemmQ40Tc(int epi, const void *qs, const void *scales, uint32_t d, uint32_t n, const void *act, uint32_t actStride, uint32_t T,
              void *out, uint32_t outStride, int numSms, cudaStream_t stream, bool pdl);
int gemmQ40TcAr(const void *qs, const void *scales, uint32_t d, uint32_t n, const void *act, uint32_t actStride, uint32_t T, void *out,
                uint32_t outStride, int numSms, cudaStream_t stream, const ArArgs &ar);   // GEMM + fused all-reduce + residual
int gemmQ40TcGrouped(int epi, const void *qs, const void *scales, uint32_t nGroups, uint32_t grpRows, uint32_t n, const void *act,
                     uint32_t actStride, uint32_t rowsTotal, uint32_t maxTokens, const int *grpCount, const int *grpOffset, void *out,
                     uint32_t outStride, int numSms, cudaStream_t stream);   // 1: shape not covered
// Mixture-of-experts feed-forward over a prompt chunk (moe_prefill.cu)
struct MoePrefillArgs {
    float *x;                     // [T][dim] residual stream, updated in place
    void *xnScratch;              // bf16 [T][dim]
    const float *norm, *gate;     // ffn rms-norm weight [dim], router gate [nExperts][dim] f32
    const void *w13Qs, *w13Sc, *w2Qs, *w2Sc;
    uint32_t T, dim, ff, nExperts, k, firstLocal, nLocal;
    float eps;
    int numSms;
    ArArgs ar;                    // nRanks > 1: partial sums are all-reduced over peer memory inside the combine kernel
};
int moePrefillFfn(const MoePrefillArgs &a, cudaStream_t stream);   // 1: shape not covered
// Launch with the programmatic-dependent-launch attribute: the kernel may start while its predecessor in the stream is still running
// and must execute griddepcontrol.wait (pdlWait) before touching anything the predecessor produces or still reads.
template <typename... KArgs, typename... Args>
inline cudaError_t launchPdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, bool pdl, Args... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = pdl ? 1 : 0;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// Prompt scoring (score.cu): log-probability of each row's target, top-1 id and its log-probability, from f32 logits rows.
constexpr uint32_t kScoreWordsPerRow = 4;   // LL words per row and source rank in the tensor-parallel record exchange
struct ScoreArgs {
    const float *logits;          // [T][ld], this rank's vocabulary slice
    uint32_t T, vocab, ld;        // rows, local vocabulary entries per row, row stride
    const int *targets;           // [T] global target ids, -1 = none
    uint32_t limit;               // global ids >= limit never win the top-1 (0 = no limit)
    uint32_t rowOffset;           // global id of local entry 0 (rank * vocab)
    float *outLogprob;            // [T] (NaN where the target is -1)
    int *outTopId;                // [T] global id
    float *outTopLogprob;         // [T]
    ArArgs ar;                    // ar.nRanks > 1: records exchanged over the peer arena, slot words [t * kScoreWordsPerRow, +4)
};
int launchScoreRows(const ScoreArgs &a, cudaStream_t stream, bool pdl);

int launchArResidual(float *x, const float *partial, uint32_t dim, uint32_t T, const ArArgs &ar, cudaStream_t stream, bool pdl = false);   // x += all-reduce(partial)
int launchRmsNormBf16(const float *x, uint32_t xStride, const float *w, void *y, uint32_t yStride, uint32_t n, float eps, uint32_t T,
                      cudaStream_t stream, bool pdl = false);

}  // namespace dl
