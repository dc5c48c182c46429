// Per-rank inference engine: owns the kernel schedule of one forward pass and the CUDA graph of the decode step.
//
// Role in the reference: NnExecutor + NnCpuDevice/NnVulkanDevice + the `start/att/ff/end` segments emitted by
// buildLlmNet (src/nn/nn-executor.cpp:45-207, src/llm.cpp:247-603) — ~26 barrier-separated ops per layer driven
// by an interpreter. Here a forward pass is a fixed sequence of 5 fused kernels per layer, chained with
// programmatic dependent launch, and the single-token step is captured once into a CUDA graph whose inputs
// (token id, position) live in device memory so the graph replays without host round trips:
// the sampling kernel writes the next token and advances the position on the device.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "engine_api.h"
#include "kernels.h"

namespace dl {

uint32_t gHiddenAct = 0;

static_assert(kApiMaxRanks == kMaxRanks, "engine_api.h and kernels.h disagree on the rank limit");

struct Buffers {   // working memory of the kernels, allocated and zeroed by dl_engine_create
    int *tokens, *pos;           // [maxBatch]
    float *x, *qkv, *z, *h, *logits;   // [maxBatch][dim | qkvDim | qDim | ff | vocab] (h: max(maxBatch, nActive) rows)
    float *attnPartial;          // [maxBatch][nHeads][nSplits][hd+2]
    unsigned int *attnCounters;  // [maxBatch][nHeads]
    int *history;                // [seqLen + 1] generated token per position (device-side log)
    // MoE scratch
    int *expertIdx;              // [maxBatch][nActive]
    float *expertWeight;         // [maxBatch][nActive]
    float *routerLogits;         // [maxBatch][nExperts]
    unsigned int *routerCounter; // [maxBatch]
    float *moeScratch;           // [nActive][dim]
    unsigned int *moeCounters;   // [256]
    // prefill (tensor-core GEMM path) buffers, maxPrefill tokens
    int *pTokens, *pPos;         // [maxPrefill]
    float *px, *pqkv;            // [maxPrefill][dim | max(qkvDim, dim)] f32; pqkv also takes the [T][dim] partial of the TP WO / W2 GEMMs
    void *pxn, *pzb, *phb;       // bf16 [maxPrefill][dim | qDim | ff]
    float *pAttnPartial;         // [maxPrefill][nHeads][hd+2]
    unsigned int *pAttnCounters; // [maxPrefill][nHeads]
    int *pTargets;               // [maxPrefill] score targets (global ids, -1 = none)
    float *pLogprob, *pTopLogprob;   // [maxPrefill] score results
    int *pTopId;                 // [maxPrefill]
    // fused arg-max scratch
    float *argVal;               // [256]
    int *argIdx;                 // [256]
    unsigned int *argCounter;    // [4]
};

struct Engine {
    EngineConfig cfg{};
    CommPtrs comm{};
    bool tp = false;             // dl_engine_set_comm was called: all-reduces run inside the kernels over the peer arena
    std::vector<LayerPtrs> layers;
    GlobalPtrs g{};
    Buffers b{};
    std::vector<void *> kCache, vCache;   // per layer, bf16 [nKvHeads][seqLen][hd]
    std::vector<void *> owned;            // device allocations freed by dl_engine_destroy
    cudaGraphExec_t decodeGraph = nullptr;
    cudaStream_t captureStream = nullptr;
    int lastError = 0;
    uint64_t *trace = nullptr;   // device buffer [maxLaunches][4] of globaltimer stamps (optional)
    uint32_t traceCap = 0;
    bool traceAllCtas = false;   // persistent kernel: every CTA records its phase stamps (skew analysis, tools/trace_mega.py --all)
    MegaLayer *megaLayers = nullptr;   // device copy of the per-layer pointer table for the persistent decode kernel
    unsigned int *megaCounter = nullptr;
    uint2 *megaX2 = nullptr;
    uint32_t megaFlags = 0;            // DL_MEGA_FLAGS (bit 0: barrier-free LL hand-off)
    uint2 *megaX = nullptr, *megaQkv = nullptr, *megaZ = nullptr, *megaH = nullptr;   // LL vectors of the persistent kernel
    unsigned int *megaSeq = nullptr;
    unsigned int *abortHost = nullptr, *abortDev = nullptr;   // mapped pinned word: device wait loops report a blown spin budget here
    uint32_t megaInflight = 2;         // DL_MEGA_INFLIGHT: producer pacing of the persistent kernel (0 = unpaced)
    uint32_t megaCtas = 0;             // DL_MEGA_CTAS: grid size override of the persistent kernel (0 = one CTA per SM)
    bool useMega = false;
    bool lastDecodeMega = false, megaFallbackWarned = false;   // did the last single-token forward run on the persistent kernel?
    // device sampler state (sampler.cu)
    unsigned long long *rngState = nullptr;
    float *probScratch = nullptr;
    float *scoreLogits = nullptr;      // [scoreMaxTokens][vocab] logits of a scored chunk (first dl_engine_score call; in `owned`)
    unsigned int *gatherEpoch = nullptr, *gatherBlockCounter = nullptr;
    float **gatherUcDev = nullptr;
    unsigned int **flagUcDev = nullptr;
    uint32_t vocabLimit = 0;     // 0 = none; otherwise the greedy arg-max ignores vocabulary rows >= vocabLimit
    bool prefillFusedAr = false; // TP prefill: GEMM + all-reduce in one kernel (DL_PREFILL_FUSED_AR=1) instead of GEMM, then all-reduce kernel
    bool tcAttn = true;          // prefill attention on tcgen05 (DL_NO_TC_ATTN=1: per-token CUDA-core kernel)
    bool fusedAttn = true, fusedArgmax = true, useTma = true;   // debugging switches (DL_NO_FUSED_ATTN / DL_NO_FUSED_ARGMAX / DL_NO_TMA)
};

#define DL_TRY(expr)                    \
    do {                                \
        const int _r = (expr);          \
        if (_r != 0) return _r;         \
    } while (0)

static EmbTable embTable(const Engine &e) {
    EmbTable t{};
    t.rowsPerRank = e.g.embRowsPerRank;
    if (t.rowsPerRank == 0) t.shard[0] = e.g.embedding;
    else for (int r = 0; r < kMaxRanks; r++) t.shard[r] = e.g.embeddingPeers[r];
    return t;
}

constexpr uint32_t kArenaMaxCtas = 256;   // logits-gather arrival counters per rank and parity

// The limits both front ends rely on: the MoE kernels route one token per launch, enginePrefill takes at most 256 tokens.
static EngineConfig applyLimits(EngineConfig c) {
    if (c.nExperts > 0) c.maxBatch = 1;
    if (c.maxPrefill > 256) c.maxPrefill = 256;
    return c;
}

struct ArenaLayout {   // byte offsets into every rank's peer arena, 256-byte aligned
    uint64_t slotsOff, flagsOff, candValOff, gatherOff, prefillSlotsOff, bytes;
};

static ArenaLayout arenaLayout(const EngineConfig &c) {
    auto align = [](uint64_t x) { return (x + 255) / 256 * 256; };
    ArenaLayout a{};
    uint64_t off = 0;
    a.slotsOff = off; off = align(off + 2ull * c.nRanks * c.maxBatch * c.dim * 8);            // LL words (f32 payload, flag) of the decode all-reduce
    a.flagsOff = off; off = align(off + 2ull * c.nRanks * kArenaMaxCtas * 4);                // logits-gather arrival counters (sampler.cu)
    a.candValOff = off; off = align(off + kMaxRanks * 8);                                    // arg-max candidates, one LL word per rank
    a.gatherOff = off; off = align(off + (uint64_t)c.maxBatch * c.vocabFull * 4);            // gathered logits (device sampler)
    a.prefillSlotsOff = off; off = align(off + 2ull * c.nRanks * c.maxPrefill * c.dim * 8);  // LL words of the prefill all-reduce
    a.bytes = off;
    return a;
}

static void fillAr(const Engine &e, ArArgs &ar, uint32_t parity) {
    const EngineConfig &c = e.cfg;
    const ArenaLayout L = arenaLayout(c);
    ar.nRanks = c.nRanks; ar.rank = c.rank; ar.parity = parity; ar.maxCtas = kArenaMaxCtas; ar.slotStride = c.maxBatch * c.dim; ar.dim = c.dim;
    ar.slotsMc = e.comm.mcArena ? (uint64_t *)((uint8_t *)e.comm.mcArena + L.slotsOff) : nullptr;
    for (uint32_t r = 0; r < c.nRanks && r < (uint32_t)kMaxRanks; r++) {
        uint8_t *base = (uint8_t *)e.comm.arena[r];
        ar.slots[r] = (uint64_t *)(base + L.slotsOff);
        ar.cand[r] = (uint64_t *)(base + L.candValOff);
    }
}

static uint32_t localVocabLimit(const Engine &e) {
    return (e.vocabLimit && e.vocabLimit < e.cfg.vocab) ? e.vocabLimit : e.cfg.vocab;
}

static int gemvSel(const Engine &e, int pro, int epi, int nb, const GemvArgs &a, int numSms, cudaStream_t stream, bool pdl) {
    if (e.cfg.wType != 0) return gemvDense((int)e.cfg.wType, pro, epi, nb, a, numSms, stream, pdl);
    if (a.ar.nRanks > 1) {   // the in-kernel all-reduce lives in the TMA kernel only
        const int r = gemvQ40Tma(pro, epi, nb, a, numSms, stream, pdl);
        return r == 1 ? -30 : r;
    }
    return e.useTma ? gemvQ40Auto(pro, epi, nb, a, numSms, stream, pdl) : gemvQ40(pro, epi, nb, a, numSms, stream, pdl);
}

// Mixture-of-experts feed-forward of one token: router -> k x (W1|W3 -> silu*up) -> k x W2; the weighted expert sum is
// *added* to `out` (the residual stream, or a zeroed partial buffer on the NCCL path), all-reduced in the epilogue if asked.
static int runMoe(Engine &e, const LayerPtrs &L, float *out, bool fusedAr, uint64_t *trace13, uint64_t *trace2, cudaStream_t stream,
                  bool pdl) {
    const EngineConfig &c = e.cfg;
    if (c.wType != 0) return -34;   // expert-indexed kernels exist for q40 matrices only
    RouterArgs ro{};
    ro.x = e.b.x; ro.normW = L.norm1; ro.gate = L.moeGate; ro.eps = c.eps; ro.dim = c.dim; ro.nExperts = c.nExperts;
    ro.k = c.nActiveExperts; ro.logits = e.b.routerLogits; ro.counter = e.b.routerCounter; ro.expertIdx = e.b.expertIdx;
    ro.expertWeight = e.b.expertWeight;
    DL_TRY(launchMoeRouter(ro, 1, stream, pdl));
    const uint32_t perSlot = c.numSms / c.nActiveExperts > 0 ? c.numSms / c.nActiveExperts : 1;
    GemvArgs a{};
    a.qs = (const uint32_t *)L.w13Qs; a.scales = (const __half *)L.w13Sc; a.d = 2 * c.ffDim; a.n = c.dim;
    a.in = e.b.x; a.inStride = c.dim; a.normW = L.norm1; a.eps = c.eps; a.out = e.b.h; a.outStride = c.ffDim; a.trace = trace13;
    a.moeCtasPerSlot = perSlot; a.kActive = c.nActiveExperts; a.expertIdx = e.b.expertIdx; a.outSlotStride = c.ffDim;
    a.expertQsStride = (uint64_t)2 * c.ffDim * (c.dim / 8); a.expertScaleStride = (uint64_t)2 * c.ffDim * (c.dim / 32);
    a.moeFirstExpert = c.moeFirstExpert; a.moeNumLocal = c.moeNumLocal;
    { const int r = gemvQ40Tma(PRO_RMSNORM_, EPI_SWIGLU_, 1, a, c.numSms, stream, pdl); if (r != 0) return r == 1 ? -31 : r; }
    a = GemvArgs{};
    a.qs = (const uint32_t *)L.w2Qs; a.scales = (const __half *)L.w2Sc; a.d = c.dim; a.n = c.ffDim;
    a.in = e.b.h; a.inStride = c.ffDim; a.inSlotStride = c.ffDim; a.out = out; a.outStride = c.dim; a.trace = trace2;
    a.moeCtasPerSlot = perSlot; a.kActive = c.nActiveExperts; a.expertIdx = e.b.expertIdx; a.expertWeight = e.b.expertWeight;
    a.expertQsStride = (uint64_t)c.dim * (c.ffDim / 8); a.expertScaleStride = (uint64_t)c.dim * (c.ffDim / 32);
    a.moeFirstExpert = c.moeFirstExpert; a.moeNumLocal = c.moeNumLocal; a.moeScratch = e.b.moeScratch; a.moeCounters = e.b.moeCounters;
    if (fusedAr) fillAr(e, a.ar, 1);
    { const int r = gemvQ40Tma(PRO_PLAIN_, EPI_MOE_DOWN_, 1, a, c.numSms, stream, pdl); if (r != 0) return r == 1 ? -32 : r; }
    return 0;
}

// One token through the persistent kernel (dense models, nb == 1). Returns 1 when the shape is not supported.
static int engineDecodeMega(Engine &e, bool greedyAdvance, cudaStream_t stream) {
    const EngineConfig &c = e.cfg;
    if (!e.megaLayers || c.nExperts > 0 || c.wType != 0) return 1;
    MegaArgs m{};
    m.layers = e.megaLayers; m.nLayers = c.nLayers; m.dim = c.dim; m.nHeads = c.nHeads; m.nKvHeads = c.nKvHeads; m.headDim = c.headDim;
    m.ffDim = c.ffDim; m.vocab = c.vocab; m.vocabFull = c.vocabFull; m.seqLen = c.seqLen; m.nSplits = c.nSplits; m.eps = c.eps;
    m.embedding = embTable(e); m.finalNorm = e.g.finalNorm; m.rope = e.g.rope;
    m.wclsQs = (const uint8_t *)e.g.wclsQs; m.wclsSc = (const uint8_t *)e.g.wclsSc;
    m.tokens = e.b.tokens; m.pos = e.b.pos; m.history = e.b.history;
    m.logits = e.b.logits; m.maxInflight = e.megaInflight;
    m.xW = e.megaX; m.xW2 = e.megaX2; m.flags = e.megaFlags; m.qkvW = e.megaQkv; m.zW = e.megaZ; m.hF = (float *)e.megaH; m.launchSeq = e.megaSeq; m.abortFlag = e.abortDev;
    m.syncNs = (e.tp && e.megaSeq) ? (unsigned long long *)(e.megaSeq + 2) : nullptr;
    m.attnPartial = e.b.attnPartial; m.attnCounters = e.b.attnCounters;
    m.argVal = e.b.argVal; m.argIdx = e.b.argIdx; m.argCounter = e.b.argCounter; m.gridCounter = e.megaCounter;
    m.rowOffsetGlobal = c.rank * c.vocab; m.greedyAdvance = greedyAdvance ? 1u : 0u; m.vocabLimit = e.vocabLimit;
    m.trace = e.trace;
    m.traceCtas = e.traceAllCtas ? c.numSms : 1u;
    m.traceStride = e.traceAllCtas ? (uint32_t)(((size_t)e.traceCap * 4) / c.numSms) : 0u;
    if (e.tp) fillAr(e, m.ar, 0);
    return launchMegaDecode(m, (int)(e.megaCtas ? e.megaCtas : c.numSms), stream);
}

// logitsMode: 0 = none (prefill chunk), 1 = logits of the last token in the batch into logits[0], 2 = all tokens
static int engineForward(Engine &e, int nb, int logitsMode, bool greedyAdvance, cudaStream_t stream) {
    const EngineConfig &c = e.cfg;
    const bool pdl = c.usePdl != 0;
    const uint32_t qDim = c.nHeads * c.headDim, kvDim = c.nKvHeads * c.headDim, qkvDim = qDim + 2 * kvDim;
    if (nb < 1 || (uint32_t)nb > c.maxBatch || (nb & (nb - 1))) return -10;
    e.lastDecodeMega = false;
    if (nb == 1 && logitsMode == 1 && e.useMega) {
        const int r = engineDecodeMega(e, greedyAdvance, stream);
        if (r != 1) { e.lastDecodeMega = r == 0; return r; }
        if (!e.megaFallbackWarned) {
            std::fprintf(stderr, "dl_engine: the persistent decode kernel cannot run this configuration (shape, shared memory or co-residency); "
                                 "using the multi-kernel path\n");
            e.megaFallbackWarned = true;
        }
    }
    uint32_t slot = 0;
    auto nextTrace = [&]() -> uint64_t * { uint64_t *t = (e.trace && slot < e.traceCap) ? e.trace + (size_t)slot * 4 : nullptr; slot++; return t; };

    DL_TRY(launchEmbedding(embTable(e), e.b.tokens, e.b.x, c.dim, c.dim, c.vocabFull, nb, stream));
    for (uint32_t l = 0; l < c.nLayers; l++) {
        const LayerPtrs &L = e.layers[l];
        GemvArgs a{};
        // 1. rmsnorm -> q80 -> QKV
        a.qs = (const uint32_t *)L.qkvQs; a.scales = (const __half *)L.qkvSc; a.d = qkvDim; a.n = c.dim;
        a.in = e.b.x; a.inStride = c.dim; a.normW = L.norm0; a.eps = c.eps; a.out = e.b.qkv; a.outStride = qkvDim; a.trace = nextTrace();
        DL_TRY(gemvSel(e, PRO_RMSNORM_, EPI_STORE_, nb, a, c.numSms, stream, pdl));
        if (nb == 1 && e.fusedAttn) {
            // 2+3. qk-norm + rope + kv append + attention in one launch
            AttnFusedArgs f{};
            f.qkv = e.b.qkv; f.pos = e.b.pos; f.rope = e.g.rope; f.qNorm = L.qNorm; f.kNorm = L.kNorm; f.eps = c.eps;
            f.kCache = (__nv_bfloat16 *)e.kCache[l]; f.vCache = (__nv_bfloat16 *)e.vCache[l];
            f.nHeads = c.nHeads; f.nKvHeads = c.nKvHeads; f.headDim = c.headDim; f.seqLen = c.seqLen; f.nSplits = c.nSplits;
            f.partial = e.b.attnPartial; f.counters = e.b.attnCounters; f.out = e.b.z; f.trace = nextTrace();
            DL_TRY(launchAttnFused(f, stream, pdl));
        } else {
            // 2. qk-norm + rope + kv write
            RopeKvArgs r{};
            r.qkv = e.b.qkv; r.qkvStride = qkvDim; r.pos = e.b.pos; r.rope = e.g.rope; r.qNorm = L.qNorm; r.kNorm = L.kNorm;
            r.eps = c.eps; r.nHeads = c.nHeads; r.nKvHeads = c.nKvHeads; r.headDim = c.headDim; r.seqLen = c.seqLen;
            r.kCache = (__nv_bfloat16 *)e.kCache[l]; r.vCache = (__nv_bfloat16 *)e.vCache[l];
            DL_TRY(launchRopeKv(r, nb, stream, pdl));
            // 3. attention
            AttnArgs t{};
            t.qkv = e.b.qkv; t.qkvStride = qkvDim; t.pos = e.b.pos; t.kCache = r.kCache; t.vCache = r.vCache;
            t.nHeads = c.nHeads; t.nKvHeads = c.nKvHeads; t.headDim = c.headDim; t.seqLen = c.seqLen; t.nSplits = c.nSplits;
            t.partial = e.b.attnPartial; t.counters = e.b.attnCounters; t.out = e.b.z; t.outStride = qDim;
            DL_TRY(launchAttnDecode(t, nb, stream, pdl));
        }
        // 4. q80 -> WO, residual add
        a = GemvArgs{};
        a.qs = (const uint32_t *)L.woQs; a.scales = (const __half *)L.woSc; a.d = c.dim; a.n = qDim;
        a.in = e.b.z; a.inStride = qDim; a.out = e.b.x; a.outStride = c.dim; a.trace = nextTrace();
        if (e.tp) fillAr(e, a.ar, 0);
        DL_TRY(gemvSel(e, PRO_PLAIN_, EPI_RESIDUAL_, nb, a, c.numSms, stream, pdl));
        if (c.nExperts > 0) {
            // 5-7. mixture of experts: router -> k x (W1|W3 -> silu*up) -> k x W2, weighted sum, residual (+ all-reduce)
            if (nb != 1) return -13;
            nextTrace();
            uint64_t *t13 = nextTrace(), *t2 = nextTrace();
            DL_TRY(runMoe(e, L, e.b.x, e.tp, t13, t2, stream, pdl));
            continue;
        }
        // 5. rmsnorm -> q80 -> W1|W3 -> silu*up
        a = GemvArgs{};
        a.qs = (const uint32_t *)L.w13Qs; a.scales = (const __half *)L.w13Sc; a.d = 2 * c.ffDim; a.n = c.dim;
        a.in = e.b.x; a.inStride = c.dim; a.normW = L.norm1; a.eps = c.eps; a.out = e.b.h; a.outStride = c.ffDim; a.trace = nextTrace();
        DL_TRY(gemvSel(e, PRO_RMSNORM_, EPI_SWIGLU_, nb, a, c.numSms, stream, pdl));
        // 6. q80 -> W2, residual add
        a = GemvArgs{};
        a.qs = (const uint32_t *)L.w2Qs; a.scales = (const __half *)L.w2Sc; a.d = c.dim; a.n = c.ffDim;
        a.in = e.b.h; a.inStride = c.ffDim; a.out = e.b.x; a.outStride = c.dim; a.trace = nextTrace();
        if (e.tp) fillAr(e, a.ar, 1);
        DL_TRY(gemvSel(e, PRO_PLAIN_, EPI_RESIDUAL_, nb, a, c.numSms, stream, pdl));
    }
    if (logitsMode != 0) {
        GemvArgs a{};
        a.qs = (const uint32_t *)e.g.wclsQs; a.scales = (const __half *)e.g.wclsSc; a.d = c.vocab; a.n = c.dim;
        a.normW = e.g.finalNorm; a.eps = c.eps; a.inStride = c.dim; a.outStride = c.vocab; a.out = e.b.logits; a.trace = nextTrace();
        if (logitsMode == 1) {
            a.in = e.b.x + (size_t)(nb - 1) * c.dim;
            int r = 1;
            if (greedyAdvance && e.fusedArgmax && c.wType == 0) {
                // logits + greedy sampling + position advance in one launch
                a.argVal = e.b.argVal; a.argIdx = e.b.argIdx; a.argCounter = e.b.argCounter;
                a.tokenOut = e.b.tokens; a.posInOut = e.b.pos; a.history = e.b.history; a.historyCap = c.seqLen;
                a.rowOffsetGlobal = c.rank * c.vocab; a.vocabLimit = e.vocabLimit;
                if (e.tp) fillAr(e, a.ar, 0);
                r = gemvQ40Tma(PRO_RMSNORM_, EPI_ARGMAX_, 1, a, c.numSms, stream, pdl);
                if (r < 0) return r;
            }
            if (r == 1) {
                // the stand-alone arg-max kernel sees this rank's vocabulary slice only: under tensor parallelism the ranks would
                // pick different (local) ids, so the non-fused route is refused there instead of silently diverging
                if (greedyAdvance && e.tp) return -33;
                a.argVal = nullptr; a.argIdx = nullptr; a.argCounter = nullptr; a.tokenOut = nullptr; a.posInOut = nullptr; a.history = nullptr;
                a.ar = ArArgs{};
                DL_TRY(gemvSel(e, PRO_RMSNORM_, EPI_STORE_, 1, a, c.numSms, stream, pdl));
                if (greedyAdvance)
                    DL_TRY(launchArgmaxAdvance(e.b.logits, localVocabLimit(e), e.b.tokens, e.b.pos, e.b.history, c.seqLen, stream, pdl));
            }
        } else {
            a.in = e.b.x;
            DL_TRY(gemvSel(e, PRO_RMSNORM_, EPI_STORE_, nb, a, c.numSms, stream, pdl));
            if (greedyAdvance) {
                if (e.tp) return -33;
                DL_TRY(launchArgmaxAdvance(e.b.logits, localVocabLimit(e), e.b.tokens, e.b.pos, e.b.history, c.seqLen, stream, pdl));
            }
        }
    }
    return 0;
}

// The layers of a prompt chunk of T <= maxPrefill tokens on the tensor-core path: writes the chunk's KV rows and leaves the final
// residual stream of every token in px.
static int prefillLayers(Engine &e, uint32_t T, uint32_t p0, cudaStream_t stream) {
    const EngineConfig &c = e.cfg;
    const GlobalPtrs &g = e.g;
    const Buffers &b = e.b;
    const bool pdl = c.usePdl != 0;   // every kernel of this chain waits (griddepcontrol.wait) before touching its predecessor's data
    const uint32_t qDim = c.nHeads * c.headDim, kvDim = c.nKvHeads * c.headDim, qkvDim = qDim + 2 * kvDim;
    if (T < 1 || T > c.maxPrefill) return -11;
    if (c.wType != 0) return -35;   // tensor-core path: q40 matrices
    const bool tp = e.tp;
    ArArgs arP{};
    if (tp) {
        fillAr(e, arP, 0);
        const uint64_t off = arenaLayout(c).prefillSlotsOff;
        arP.slotStride = c.maxPrefill * c.dim;
        for (uint32_t r = 0; r < c.nRanks; r++) arP.slots[r] = (uint64_t *)((uint8_t *)e.comm.arena[r] + off);
        arP.slotsMc = e.comm.mcArena ? (uint64_t *)((uint8_t *)e.comm.mcArena + off) : nullptr;
    }
    DL_TRY(launchEmbedding(embTable(e), b.pTokens, b.px, c.dim, c.dim, c.vocabFull, (int)T, stream));
    for (uint32_t l = 0; l < c.nLayers; l++) {
        const LayerPtrs &L = e.layers[l];
        DL_TRY(launchRmsNormBf16(b.px, c.dim, L.norm0, b.pxn, c.dim, c.dim, c.eps, T, stream, pdl));
        DL_TRY(gemmQ40Tc(GEPI_STORE_F32_, L.qkvQs, L.qkvSc, qkvDim, c.dim, b.pxn, c.dim, T, b.pqkv, qkvDim, c.numSms, stream, pdl));
        RopeKvArgs r{};
        r.qkv = b.pqkv; r.qkvStride = qkvDim; r.pos = b.pPos; r.rope = g.rope; r.qNorm = L.qNorm; r.kNorm = L.kNorm;
        r.eps = c.eps; r.nHeads = c.nHeads; r.nKvHeads = c.nKvHeads; r.headDim = c.headDim; r.seqLen = c.seqLen;
        r.kCache = (__nv_bfloat16 *)e.kCache[l]; r.vCache = (__nv_bfloat16 *)e.vCache[l];
        DL_TRY(launchRopeKv(r, (int)T, stream, pdl));
        int attnRc = 1;
        if (e.tcAttn) {
            // tensor-core attention over the whole chunk: the tokens of a chunk sit at consecutive positions p0 .. p0 + T - 1
            AttnPrefillArgs ap{};
            ap.qkv = b.pqkv; ap.qkvStride = qkvDim; ap.T = T; ap.p0 = p0; ap.nHeads = c.nHeads; ap.nKvHeads = c.nKvHeads;
            ap.headDim = c.headDim; ap.seqLen = c.seqLen; ap.kCache = r.kCache; ap.vCache = r.vCache;
            ap.out = (__nv_bfloat16 *)b.pzb; ap.outStride = qDim;
            attnRc = launchAttnPrefillTc(ap, stream, pdl);
            if (attnRc < 0) return attnRc;
        }
        if (attnRc == 1) {
            AttnArgs t{};
            t.qkv = b.pqkv; t.qkvStride = qkvDim; t.pos = b.pPos; t.kCache = r.kCache; t.vCache = r.vCache;
            t.nHeads = c.nHeads; t.nKvHeads = c.nKvHeads; t.headDim = c.headDim; t.seqLen = c.seqLen; t.nSplits = 1;
            t.partial = b.pAttnPartial; t.counters = b.pAttnCounters; t.out = nullptr; t.outStride = qDim; t.outBf16 = (__nv_bfloat16 *)b.pzb;
            DL_TRY(launchAttnDecode(t, (int)T, stream, pdl));
        }
        // tensor parallel: partial product into the (now free) qkv buffer with all SMs / split-K, then all-reduce + residual over
        // peer memory as its own kernel (DL_PREFILL_FUSED_AR=1: the one-kernel GEMM + all-reduce epilogue instead)
        if (tp && !e.prefillFusedAr) {
            arP.parity = 0;
            DL_TRY(gemmQ40Tc(GEPI_STORE_F32_, L.woQs, L.woSc, c.dim, qDim, b.pzb, qDim, T, b.pqkv, c.dim, c.numSms, stream, pdl));
            DL_TRY(launchArResidual(b.px, b.pqkv, c.dim, T, arP, stream, pdl));
        } else if (tp) { arP.parity = 0; DL_TRY(gemmQ40TcAr(L.woQs, L.woSc, c.dim, qDim, b.pzb, qDim, T, b.px, c.dim, c.numSms, stream, arP)); }
        else DL_TRY(gemmQ40Tc(GEPI_RESIDUAL_, L.woQs, L.woSc, c.dim, qDim, b.pzb, qDim, T, b.px, c.dim, c.numSms, stream, pdl));
        if (c.nExperts > 0) {
            // mixture of experts: route the whole chunk, sort the (token, expert) pairs, grouped tensor-core GEMMs, weighted combine
            MoePrefillArgs mo{};
            mo.x = b.px; mo.xnScratch = b.pxn; mo.norm = L.norm1; mo.gate = L.moeGate; mo.w13Qs = L.w13Qs; mo.w13Sc = L.w13Sc;
            mo.w2Qs = L.w2Qs; mo.w2Sc = L.w2Sc; mo.T = T; mo.dim = c.dim; mo.ff = c.ffDim; mo.nExperts = c.nExperts; mo.k = c.nActiveExperts;
            mo.firstLocal = c.moeFirstExpert; mo.nLocal = c.moeNumLocal; mo.eps = c.eps; mo.numSms = (int)c.numSms;
            if (tp) { arP.parity = 1; mo.ar = arP; }
            const int mr = moePrefillFfn(mo, stream);
            if (mr != 0) return mr == 1 ? -36 : mr;
            continue;
        }
        DL_TRY(launchRmsNormBf16(b.px, c.dim, L.norm1, b.pxn, c.dim, c.dim, c.eps, T, stream, pdl));
        DL_TRY(gemmQ40Tc(GEPI_SWIGLU_BF16_, L.w13Qs, L.w13Sc, 2 * c.ffDim, c.dim, b.pxn, c.dim, T, b.phb, c.ffDim, c.numSms, stream, pdl));
        if (tp && !e.prefillFusedAr) {
            arP.parity = 1;
            DL_TRY(gemmQ40Tc(GEPI_STORE_F32_, L.w2Qs, L.w2Sc, c.dim, c.ffDim, b.phb, c.ffDim, T, b.pqkv, c.dim, c.numSms, stream, pdl));
            DL_TRY(launchArResidual(b.px, b.pqkv, c.dim, T, arP, stream, pdl));
        } else if (tp) { arP.parity = 1; DL_TRY(gemmQ40TcAr(L.w2Qs, L.w2Sc, c.dim, c.ffDim, b.phb, c.ffDim, T, b.px, c.dim, c.numSms, stream, arP)); }
        else DL_TRY(gemmQ40Tc(GEPI_RESIDUAL_, L.w2Qs, L.w2Sc, c.dim, c.ffDim, b.phb, c.ffDim, T, b.px, c.dim, c.numSms, stream, pdl));
    }
    return 0;
}

// Prompt chunk of T <= maxPrefill tokens on the tensor-core path. Logits (optional) are produced for the last token.
static int enginePrefill(Engine &e, uint32_t T, uint32_t p0, int wantLogits, cudaStream_t stream) {
    const EngineConfig &c = e.cfg;
    const GlobalPtrs &g = e.g;
    const Buffers &b = e.b;
    DL_TRY(prefillLayers(e, T, p0, stream));
    if (wantLogits) {
        GemvArgs a{};
        a.qs = (const uint32_t *)g.wclsQs; a.scales = (const __half *)g.wclsSc; a.d = c.vocab; a.n = c.dim;
        a.normW = g.finalNorm; a.eps = c.eps; a.inStride = c.dim; a.outStride = c.vocab; a.out = b.logits;
        a.in = b.px + (size_t)(T - 1) * c.dim;
        DL_TRY(gemvSel(e, PRO_RMSNORM_, EPI_STORE_, 1, a, c.numSms, stream, false));
    }
    return 0;
}

// Tokens per dl_engine_score call: the chunk limit of the prefill chain, and under tensor parallelism also the rows whose score
// records fit into one parity of the decode all-reduce slots (maxBatch * dim words per source rank; maxBatch is 1 for MoE models).
static uint32_t scoreMaxTokens(const EngineConfig &c) {
    if (c.nRanks <= 1) return c.maxPrefill;
    return std::min(c.maxPrefill, c.maxBatch * c.dim / kScoreWordsPerRow);
}

// Prompt chunk on the tensor-core path, then the logits of all T tokens and their scores against the targets staged in pTargets.
static int engineScore(Engine &e, uint32_t T, uint32_t p0, cudaStream_t stream) {
    const EngineConfig &c = e.cfg;
    const Buffers &b = e.b;
    const bool pdl = c.usePdl != 0;
    const uint32_t maxT = scoreMaxTokens(c);
    if (T < 1 || T > maxT) return -11;
    if (c.wType != 0) return -35;
    if (c.nRanks > 1 && !e.tp) return -37;
    if (!e.scoreLogits) {   // [maxScore][vocab] f32, allocated on the first call so that engines that never score keep their footprint
        void *p = nullptr;
        DL_CUDA_CHECK(cudaMalloc(&p, (size_t)maxT * c.vocab * sizeof(float)));
        e.owned.push_back(p);
        e.scoreLogits = (float *)p;
    }
    DL_TRY(prefillLayers(e, T, p0, stream));
    DL_TRY(launchRmsNormBf16(b.px, c.dim, e.g.finalNorm, b.pxn, c.dim, c.dim, c.eps, T, stream, pdl));
    DL_TRY(gemmQ40Tc(GEPI_STORE_F32_, e.g.wclsQs, e.g.wclsSc, c.vocab, c.dim, b.pxn, c.dim, T, e.scoreLogits, c.vocab, c.numSms, stream, pdl));
    ScoreArgs s{};
    s.logits = e.scoreLogits; s.T = T; s.vocab = c.vocab; s.ld = c.vocab; s.targets = b.pTargets; s.limit = e.vocabLimit;
    s.rowOffset = c.rank * c.vocab; s.outLogprob = b.pLogprob; s.outTopId = b.pTopId; s.outTopLogprob = b.pTopLogprob;
    // The records travel through parity 1 of the decode all-reduce slots. Every use of a slot word is a write by the source rank
    // followed by a read-and-reset by the owning rank, so a write must not land before the previous use's reset. Rank A writes
    // rank B's words in this kernel only after its own prefill all-reduces of this chunk, which read words that B wrote after
    // finishing, in stream order, whatever B ran before (a decode step's W2 / MoE all-reduce on parity 1, or the previous
    // chunk's score kernel): those resets are done. In the other direction, the next user of parity 1 on A (a decode step's W2
    // or MoE all-reduce, or the next chunk's score) comes after a parity-0 WO all-reduce or the next chunk's prefill all-reduces,
    // which need B's contribution, written after B's score kernel and its resets completed.
    if (e.tp) fillAr(e, s.ar, 1);
    return launchScoreRows(s, stream, pdl);
}

// Allocates and zeroes the working buffers and KV caches on the current device, finished before it returns: a forward may
// read cache rows that no kernel has written yet.
static bool allocBuffers(Engine &e) {
    const EngineConfig &c = e.cfg;
    bool ok = true;
    auto zeroed = [&](size_t bytes) -> void * {
        void *p = nullptr;
        if (!ok || bytes == 0) return nullptr;
        if (cudaMalloc(&p, bytes) != cudaSuccess) { ok = false; return nullptr; }
        e.owned.push_back(p);
        ok = cudaMemset(p, 0, bytes) == cudaSuccess;
        return p;
    };
    const size_t mb = c.maxBatch, mp = c.maxPrefill, dim = c.dim, ff = c.ffDim, heads = c.nHeads, hd = c.headDim;
    const size_t kAct = std::max(1u, c.nActiveExperts), qDim = heads * hd, qkvDim = qDim + 2 * (size_t)c.nKvHeads * hd;
    Buffers &b = e.b;
    b.tokens = (int *)zeroed(mb * 4); b.pos = (int *)zeroed(mb * 4);
    b.x = (float *)zeroed(mb * dim * 4); b.qkv = (float *)zeroed(mb * qkvDim * 4); b.z = (float *)zeroed(mb * qDim * 4);
    b.h = (float *)zeroed(std::max(mb, kAct) * ff * 4); b.logits = (float *)zeroed(mb * c.vocab * 4);
    b.attnPartial = (float *)zeroed(mb * heads * c.nSplits * (hd + 2) * 4); b.attnCounters = (unsigned int *)zeroed(mb * heads * 4);
    b.history = (int *)zeroed(((size_t)c.seqLen + 1) * 4);
    b.expertIdx = (int *)zeroed(mb * kAct * 4); b.expertWeight = (float *)zeroed(mb * kAct * 4);
    b.routerLogits = (float *)zeroed(mb * std::max(1u, c.nExperts) * 4); b.routerCounter = (unsigned int *)zeroed(mb * 4);
    b.moeScratch = (float *)zeroed(kAct * dim * 4); b.moeCounters = (unsigned int *)zeroed(256 * 4);
    b.pTokens = (int *)zeroed(mp * 4); b.pPos = (int *)zeroed(mp * 4);
    b.px = (float *)zeroed(mp * dim * 4); b.pqkv = (float *)zeroed(mp * std::max(qkvDim, dim) * 4);
    b.pxn = zeroed(mp * dim * 2); b.pzb = zeroed(mp * qDim * 2); b.phb = zeroed(mp * ff * 2);
    b.pAttnPartial = (float *)zeroed(mp * heads * (hd + 2) * 4); b.pAttnCounters = (unsigned int *)zeroed(mp * heads * 4);
    b.pTargets = (int *)zeroed(mp * 4); b.pLogprob = (float *)zeroed(mp * 4); b.pTopId = (int *)zeroed(mp * 4);
    b.pTopLogprob = (float *)zeroed(mp * 4);
    b.argVal = (float *)zeroed(256 * 4); b.argIdx = (int *)zeroed(256 * 4); b.argCounter = (unsigned int *)zeroed(4 * 4);
    for (uint32_t l = 0; l < c.nLayers; l++) {
        e.kCache.push_back(zeroed((size_t)c.nKvHeads * c.seqLen * hd * 2));
        e.vCache.push_back(zeroed((size_t)c.nKvHeads * c.seqLen * hd * 2));
    }
    return ok && cudaDeviceSynchronize() == cudaSuccess;
}

}  // namespace dl

using dl::Engine;

DL_EXPORT void *dl_engine_create(const dl::EngineConfig *cfg) {
    Engine *e = new Engine();
    e->cfg = dl::applyLimits(*cfg);
    dl::gHiddenAct = cfg->hiddenAct;
    e->layers.resize(cfg->nLayers);
    e->fusedAttn = std::getenv("DL_NO_FUSED_ATTN") == nullptr;
    e->fusedArgmax = std::getenv("DL_NO_FUSED_ARGMAX") == nullptr;
    e->useTma = std::getenv("DL_NO_TMA") == nullptr;
    e->tcAttn = std::getenv("DL_NO_TC_ATTN") == nullptr;
    e->prefillFusedAr = std::getenv("DL_PREFILL_FUSED_AR") != nullptr;
    if (e->cfg.numSms == 0) {
        int dev = 0, sms = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        e->cfg.numSms = (uint32_t)sms;
    }
    if (e->cfg.nSplits == 0) e->cfg.nSplits = std::max(1u, std::min(32u, 2 * e->cfg.numSms / std::max(1u, e->cfg.nHeads)));
    if (!dl::allocBuffers(*e)) {
        dl_engine_destroy(e);
        return nullptr;
    }
    return e;
}

DL_EXPORT void dl_engine_destroy(void *h) {
    Engine *e = (Engine *)h;
    if (!e) return;
    if (e->decodeGraph) cudaGraphExecDestroy(e->decodeGraph);
    if (e->captureStream) cudaStreamDestroy(e->captureStream);
    if (e->megaLayers) cudaFree(e->megaLayers);
    if (e->megaCounter) cudaFree(e->megaCounter);
    for (void *q : {(void *)e->megaX, (void *)e->megaX2, (void *)e->megaQkv, (void *)e->megaZ, (void *)e->megaH, (void *)e->megaSeq}) if (q) cudaFree(q);
    if (e->abortHost) cudaFreeHost(e->abortHost);
    for (void *p : e->owned) cudaFree(p);
    delete e;
}

DL_EXPORT int dl_engine_set_layer(void *h, uint32_t layer, const dl::LayerPtrs *p) {
    Engine *e = (Engine *)h;
    if (layer >= e->layers.size()) return -1;
    e->layers[layer] = *p;
    return 0;
}

DL_EXPORT int dl_engine_set_globals(void *h, const dl::GlobalPtrs *p) {
    ((Engine *)h)->g = *p;
    return 0;
}

DL_EXPORT int dl_engine_get_config(void *h, dl::EngineConfig *cfg) {
    *cfg = ((Engine *)h)->cfg;
    return 0;
}

DL_EXPORT int dl_engine_buffers(void *h, dl::EngineBuffers *out) {
    const Engine *e = (Engine *)h;
    const dl::Buffers &b = e->b;
    *out = dl::EngineBuffers{b.tokens, b.pos, b.history, b.logits, b.x, b.pTokens, b.pPos, e->kCache.data(), e->vCache.data(),
                             b.pTargets, b.pLogprob, b.pTopId, b.pTopLogprob};
    return 0;
}

DL_EXPORT uint32_t dl_engine_score_max_tokens(void *h) { return dl::scoreMaxTokens(((Engine *)h)->cfg); }

DL_EXPORT size_t dl_engine_arena_bytes(const dl::EngineConfig *cfg) { return dl::arenaLayout(dl::applyLimits(*cfg)).bytes; }

// Uploads the per-layer pointer table and switches single-token forwards to the persistent kernel.
DL_EXPORT int dl_engine_enable_mega(void *h, int enable) {
    Engine *e = (Engine *)h;
    if (enable && !e->megaLayers) {
        std::vector<dl::MegaLayer> tab(e->layers.size());
        for (size_t l = 0; l < tab.size(); l++) {
            const dl::LayerPtrs &L = e->layers[l];
            dl::MegaLayer &m = tab[l];
            m.qkvQs = (const uint8_t *)L.qkvQs; m.qkvSc = (const uint8_t *)L.qkvSc; m.woQs = (const uint8_t *)L.woQs; m.woSc = (const uint8_t *)L.woSc;
            m.w13Qs = (const uint8_t *)L.w13Qs; m.w13Sc = (const uint8_t *)L.w13Sc; m.w2Qs = (const uint8_t *)L.w2Qs; m.w2Sc = (const uint8_t *)L.w2Sc;
            m.norm0 = L.norm0; m.norm1 = L.norm1; m.qNorm = L.qNorm; m.kNorm = L.kNorm;
            m.kCache = (__nv_bfloat16 *)e->kCache[l]; m.vCache = (__nv_bfloat16 *)e->vCache[l];
        }
        DL_CUDA_CHECK(cudaMalloc(&e->megaLayers, tab.size() * sizeof(dl::MegaLayer)));
        DL_CUDA_CHECK(cudaMemcpy(e->megaLayers, tab.data(), tab.size() * sizeof(dl::MegaLayer), cudaMemcpyHostToDevice));
        DL_CUDA_CHECK(cudaMalloc(&e->megaCounter, 256));
        DL_CUDA_CHECK(cudaMemset(e->megaCounter, 0, 256));
        const dl::EngineConfig &c = e->cfg;
        const size_t qDim = (size_t)c.nHeads * c.headDim, qkvDim = qDim + 2 * (size_t)c.nKvHeads * c.headDim;
        auto allocW = [](uint2 **p, size_t n) {
            const size_t bytes = (n + 8) * sizeof(uint2);
            if (cudaMalloc(p, bytes) != cudaSuccess) return false;
            return cudaMemset(*p, 0, bytes) == cudaSuccess;
        };
        if (!allocW(&e->megaX, c.dim) || !allocW(&e->megaX2, c.dim) || !allocW(&e->megaQkv, qkvDim) || !allocW(&e->megaZ, qDim) || !allocW(&e->megaH, c.ffDim)) return -41;
        DL_CUDA_CHECK(cudaMalloc(&e->megaSeq, 256));
        const unsigned int one = 1;
        DL_CUDA_CHECK(cudaMemset(e->megaSeq, 0, 256));
        DL_CUDA_CHECK(cudaMemcpy(e->megaSeq, &one, sizeof(one), cudaMemcpyHostToDevice));   // epochs start at 1024: never equal to the zeroed words
        if (!e->abortHost) {
            DL_CUDA_CHECK(cudaHostAlloc((void **)&e->abortHost, 64, cudaHostAllocMapped));
            std::memset(e->abortHost, 0, 64);
            DL_CUDA_CHECK(cudaHostGetDevicePointer((void **)&e->abortDev, e->abortHost, 0));
        }
        if (const char *g = std::getenv("DL_MEGA_CTAS")) e->megaCtas = (uint32_t)std::atoi(g);
        if (const char *g = std::getenv("DL_MEGA_FLAGS")) e->megaFlags = (uint32_t)std::atoi(g);
        if (const char *g = std::getenv("DL_MEGA_INFLIGHT")) e->megaInflight = (uint32_t)std::atoi(g);
    }
    e->useMega = enable != 0;
    return 0;
}

DL_EXPORT int dl_engine_set_vocab_limit(void *h, uint32_t limit) {
    Engine *e = (Engine *)h;
    if (e->vocabLimit != limit && e->decodeGraph) { cudaGraphExecDestroy(e->decodeGraph); e->decodeGraph = nullptr; }   // the limit is baked into the captured launch
    e->vocabLimit = limit;
    return 0;
}

// Nanoseconds the persistent kernel (CTA 0) has spent waiting for peer ranks inside the fused all-reduce epilogues since engine
// creation (host-mapped counter: readable without a device synchronisation; exact after the stream has been synchronised).
DL_EXPORT unsigned long long dl_engine_sync_ns(void *h) {
    Engine *e = (Engine *)h;
    unsigned long long v = 0;
    if (e->megaSeq && cudaMemcpy(&v, e->megaSeq + 2, sizeof(v), cudaMemcpyDeviceToHost) != cudaSuccess) return 0ull;
    return v;
}

// 1 when a device-side wait loop gave up (dead peer rank, CTA that never became resident): the results of that step are invalid.
DL_EXPORT int dl_engine_aborted(void *h) {
    Engine *e = (Engine *)h;
    return (e->abortHost && *e->abortHost) ? 1 : 0;
}

// Seeds the device-resident xorshift* generator (same stream of coins as the host Sampler for the same seed) and allocates the
// sampler scratch. Under tensor parallelism every rank must call this with the same seed.
DL_EXPORT int dl_engine_sampler_seed(void *h, unsigned long long seed) {
    Engine *e = (Engine *)h;
    const dl::EngineConfig &c = e->cfg;
    if (!e->rngState) {
        DL_CUDA_CHECK(cudaMalloc(&e->rngState, 64));
        DL_CUDA_CHECK(cudaMalloc(&e->probScratch, ((size_t)c.vocab * (c.nRanks ? c.nRanks : 1) + 16) * sizeof(float)));
        DL_CUDA_CHECK(cudaMalloc(&e->gatherEpoch, 64));
        DL_CUDA_CHECK(cudaMemset(e->gatherEpoch, 0, 64));
        DL_CUDA_CHECK(cudaMalloc(&e->gatherBlockCounter, 64));
        DL_CUDA_CHECK(cudaMemset(e->gatherBlockCounter, 0, 64));
        if (e->tp) {
            const dl::ArenaLayout L = dl::arenaLayout(c);
            float *g[dl::kApiMaxRanks] = {};
            unsigned int *f[dl::kApiMaxRanks] = {};
            for (uint32_t r = 0; r < c.nRanks; r++) {
                g[r] = (float *)((uint8_t *)e->comm.arena[r] + L.gatherOff);
                f[r] = (unsigned int *)((uint8_t *)e->comm.arena[r] + L.flagsOff);
            }
            DL_CUDA_CHECK(cudaMalloc(&e->gatherUcDev, sizeof(g)));
            DL_CUDA_CHECK(cudaMalloc(&e->flagUcDev, sizeof(f)));
            DL_CUDA_CHECK(cudaMemcpy(e->gatherUcDev, g, sizeof(g), cudaMemcpyHostToDevice));
            DL_CUDA_CHECK(cudaMemcpy(e->flagUcDev, f, sizeof(f), cudaMemcpyHostToDevice));
        }
    }
    if (seed == 0) seed = 0x9E3779B97F4A7C15ull;   // xorshift state must not be zero
    DL_CUDA_CHECK(cudaMemcpy(e->rngState, &seed, sizeof(seed), cudaMemcpyHostToDevice));
    return 0;
}

// Samples the next token from the logits of the last forward (logitsMode 1) on the device: tokens[0] <- sample, pos[0]++, history.
// Tensor parallel: the vocabulary slices are first gathered into every rank's arena (peer / multicast stores, no NCCL); every rank
// then draws the same token from its own copy of the generator.
DL_EXPORT int dl_engine_sample(void *h, float temperature, float topp, cudaStream_t stream) {
    Engine *e = (Engine *)h;
    const dl::EngineConfig &c = e->cfg;
    if (!e->rngState) return -50;
    const uint32_t nR = e->tp ? c.nRanks : 1;
    const uint32_t full = c.vocab * nR;
    const uint32_t n = (e->vocabLimit && e->vocabLimit < full) ? e->vocabLimit : full;
    if (nR == 1)
        return dl::launchSample(e->b.logits, e->probScratch, n, temperature, topp, e->rngState, e->b.tokens, e->b.pos, e->b.history, c.seqLen,
                                nullptr, nullptr, 1, stream);
    const dl::ArenaLayout L = dl::arenaLayout(c);
    uint8_t *mine = (uint8_t *)e->comm.arena[c.rank];
    float *gatherLocal = (float *)(mine + L.gatherOff);
    unsigned int *flagLocal = (unsigned int *)(mine + L.flagsOff);
    float *gatherMc = e->comm.mcArena ? (float *)((uint8_t *)e->comm.mcArena + L.gatherOff) : nullptr;
    unsigned int *flagMc = e->comm.mcArena ? (unsigned int *)((uint8_t *)e->comm.mcArena + L.flagsOff) : nullptr;
    DL_TRY(dl::launchLogitsGather(e->b.logits, c.vocab, c.rank, nR, gatherMc, e->gatherUcDev, flagMc, e->flagUcDev, e->gatherBlockCounter, stream));
    return dl::launchSample(gatherLocal, e->probScratch, n, temperature, topp, e->rngState, e->b.tokens, e->b.pos, e->b.history, c.seqLen, flagLocal,
                            e->gatherEpoch, nR, stream);
}

DL_EXPORT int dl_engine_set_comm(void *h, const dl::CommPtrs *p) {
    Engine *e = (Engine *)h;
    e->comm = *p;
    e->tp = e->cfg.nRanks > 1;
    return 0;
}

DL_EXPORT int dl_engine_set_trace(void *h, uint64_t *buf, uint32_t capLaunches) {
    ((Engine *)h)->trace = buf;
    ((Engine *)h)->traceCap = capLaunches;
    return 0;
}

DL_EXPORT int dl_engine_set_trace_all(void *h, int allCtas) {
    ((Engine *)h)->traceAllCtas = allCtas != 0;
    return 0;
}

DL_EXPORT int dl_engine_mega_active(void *h) { return ((Engine *)h)->lastDecodeMega ? 1 : 0; }

DL_EXPORT int dl_engine_forward(void *h, int nb, int logitsMode, int greedyAdvance, cudaStream_t stream) {
    return dl::engineForward(*(Engine *)h, nb, logitsMode, greedyAdvance != 0, stream);
}

// Library-collective building blocks (decode path, nb tokens): the same kernels, but the tensor-parallel partial products
// are *stored* into `ybuf` instead of being all-reduced in the epilogue; the caller all-reduces ybuf with NCCL and adds it
// to x. Used (a) as the NCCL baseline the fused kernels are measured against, (b) as the execution path when ranks do not
// share an NVLink/IPC domain (multi-node) and (c) for dense f32/f16 weight files under tensor parallelism.
//   part 0: embedding              part 1: QKV + attention + WO -> ybuf
//   part 2: feed-forward -> ybuf   part 3: logits of the last token (local vocabulary slice)   part 4: logits of all nb tokens
DL_EXPORT int dl_engine_forward_part(void *h, int nb, uint32_t layer, int part, float *ybuf, cudaStream_t stream) {
    Engine &e = *(Engine *)h;
    const dl::EngineConfig &c = e.cfg;
    const uint32_t qDim = c.nHeads * c.headDim, kvDim = c.nKvHeads * c.headDim, qkvDim = qDim + 2 * kvDim;
    if (nb < 1 || (uint32_t)nb > c.maxBatch || (nb & (nb - 1))) return -10;
    if (part == 0) return dl::launchEmbedding(embTable(e), e.b.tokens, e.b.x, c.dim, c.dim, c.vocabFull, nb, stream);
    if (part == 3 || part == 4) {
        dl::GemvArgs a{};
        a.qs = (const uint32_t *)e.g.wclsQs; a.scales = (const __half *)e.g.wclsSc; a.d = c.vocab; a.n = c.dim;
        a.normW = e.g.finalNorm; a.eps = c.eps; a.inStride = c.dim; a.outStride = c.vocab; a.out = e.b.logits;
        a.in = part == 3 ? e.b.x + (size_t)(nb - 1) * c.dim : e.b.x;
        return dl::gemvSel(e, dl::PRO_RMSNORM_, dl::EPI_STORE_, part == 3 ? 1 : nb, a, c.numSms, stream, false);
    }
    if (layer >= c.nLayers) return -1;
    const dl::LayerPtrs &L = e.layers[layer];
    dl::GemvArgs a{};
    if (part == 1) {
        a.qs = (const uint32_t *)L.qkvQs; a.scales = (const __half *)L.qkvSc; a.d = qkvDim; a.n = c.dim;
        a.in = e.b.x; a.inStride = c.dim; a.normW = L.norm0; a.eps = c.eps; a.out = e.b.qkv; a.outStride = qkvDim;
        DL_TRY(dl::gemvSel(e, dl::PRO_RMSNORM_, dl::EPI_STORE_, nb, a, c.numSms, stream, false));
        dl::RopeKvArgs r{};
        r.qkv = e.b.qkv; r.qkvStride = qkvDim; r.pos = e.b.pos; r.rope = e.g.rope; r.qNorm = L.qNorm; r.kNorm = L.kNorm;
        r.eps = c.eps; r.nHeads = c.nHeads; r.nKvHeads = c.nKvHeads; r.headDim = c.headDim; r.seqLen = c.seqLen;
        r.kCache = (__nv_bfloat16 *)e.kCache[layer]; r.vCache = (__nv_bfloat16 *)e.vCache[layer];
        DL_TRY(dl::launchRopeKv(r, nb, stream, false));
        dl::AttnArgs t{};
        t.qkv = e.b.qkv; t.qkvStride = qkvDim; t.pos = e.b.pos; t.kCache = r.kCache; t.vCache = r.vCache;
        t.nHeads = c.nHeads; t.nKvHeads = c.nKvHeads; t.headDim = c.headDim; t.seqLen = c.seqLen; t.nSplits = c.nSplits;
        t.partial = e.b.attnPartial; t.counters = e.b.attnCounters; t.out = e.b.z; t.outStride = qDim;
        DL_TRY(dl::launchAttnDecode(t, nb, stream, false));
        a = dl::GemvArgs{};
        a.qs = (const uint32_t *)L.woQs; a.scales = (const __half *)L.woSc; a.d = c.dim; a.n = qDim;
        a.in = e.b.z; a.inStride = qDim; a.out = ybuf; a.outStride = c.dim;
        return dl::gemvSel(e, dl::PRO_PLAIN_, dl::EPI_STORE_, nb, a, c.numSms, stream, false);
    }
    if (part == 2 && c.nExperts > 0) {
        if (nb != 1) return -13;
        DL_CUDA_CHECK(cudaMemsetAsync(ybuf, 0, (size_t)c.dim * sizeof(float), stream));
        return dl::runMoe(e, L, ybuf, false, nullptr, nullptr, stream, false);
    }
    if (part == 2) {
        a.qs = (const uint32_t *)L.w13Qs; a.scales = (const __half *)L.w13Sc; a.d = 2 * c.ffDim; a.n = c.dim;
        a.in = e.b.x; a.inStride = c.dim; a.normW = L.norm1; a.eps = c.eps; a.out = e.b.h; a.outStride = c.ffDim;
        DL_TRY(dl::gemvSel(e, dl::PRO_RMSNORM_, dl::EPI_SWIGLU_, nb, a, c.numSms, stream, false));
        a = dl::GemvArgs{};
        a.qs = (const uint32_t *)L.w2Qs; a.scales = (const __half *)L.w2Sc; a.d = c.dim; a.n = c.ffDim;
        a.in = e.b.h; a.inStride = c.ffDim; a.out = ybuf; a.outStride = c.dim;
        return dl::gemvSel(e, dl::PRO_PLAIN_, dl::EPI_STORE_, nb, a, c.numSms, stream, false);
    }
    return -2;
}

DL_EXPORT int dl_engine_prefill(void *h, uint32_t T, uint32_t p0, int wantLogits, cudaStream_t stream) {
    return dl::enginePrefill(*(Engine *)h, T, p0, wantLogits, stream);
}

DL_EXPORT int dl_engine_score(void *h, uint32_t T, uint32_t p0, cudaStream_t stream) {
    return dl::engineScore(*(Engine *)h, T, p0, stream);
}

// Captures one greedy decode step (forward of 1 token + argmax + position advance) into a graph.
DL_EXPORT int dl_engine_capture_decode(void *h) {
    Engine *e = (Engine *)h;
    if (!e->captureStream) DL_CUDA_CHECK(cudaStreamCreateWithFlags(&e->captureStream, cudaStreamNonBlocking));
    if (e->decodeGraph) { cudaGraphExecDestroy(e->decodeGraph); e->decodeGraph = nullptr; }
    DL_CUDA_CHECK(cudaStreamBeginCapture(e->captureStream, cudaStreamCaptureModeThreadLocal));
    const int r = dl::engineForward(*e, 1, 1, true, e->captureStream);
    cudaGraph_t graph = nullptr;
    const cudaError_t endErr = cudaStreamEndCapture(e->captureStream, &graph);
    if (r != 0) { if (graph) cudaGraphDestroy(graph); return r; }
    DL_CUDA_CHECK(endErr);
    DL_CUDA_CHECK(cudaGraphInstantiate(&e->decodeGraph, graph, 0));
    cudaGraphDestroy(graph);
    return 0;
}

// Replays the captured step `nSteps` times back to back on `stream` (no host sync in between).
DL_EXPORT int dl_engine_decode_graph(void *h, int nSteps, cudaStream_t stream) {
    Engine *e = (Engine *)h;
    if (!e->decodeGraph) return -20;
    for (int i = 0; i < nSteps; i++) DL_CUDA_CHECK(cudaGraphLaunch(e->decodeGraph, stream));
    return 0;
}
