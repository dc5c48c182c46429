// C ABI of the per-rank engine in _cuda.so: plain structs + extern "C" entry points. Shared by engine.cu, the ctypes mirror in
// distributed_llama_b200/ops/cuda_lib.py and the native (Python-free) runtime under csrc/app/.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

namespace dl {

constexpr int kApiMaxRanks = 8;

struct EngineConfig {   // mirrored by ctypes in distributed_llama_b200/ops/cuda_lib.py
    uint32_t dim, nLayers, nHeads, nKvHeads, headDim, ffDim, vocab, seqLen;   // per-rank (sliced) head/ff/vocab counts
    uint32_t nExperts, nActiveExperts;
    uint32_t maxBatch;       // tokens per forward on the GEMV path (mixture of experts: always 1)
    uint32_t nSplits;        // attention KV splits (0: max(1, min(32, 2 * numSms / nHeads)))
    uint32_t rank, nRanks;
    uint32_t numSms;         // 0: the current device's SM count
    float eps;
    uint32_t usePdl;
    uint32_t moeFirstExpert, moeNumLocal;   // experts held by this rank (expert parallelism); TP mode: 0, nExperts
    uint32_t wType;          // matrix storage: 0 = q40 device layout, 1 = dense f32, 2 = dense f16 (gemv_dense.cu)
    uint32_t hiddenAct;      // gate activation: 0 = SiLU, 1 = GELU (tanh form) — the `.m` header's hidden_act
    uint32_t vocabFull;      // rows of the whole embedding table
    uint32_t maxPrefill;     // tokens per chunk on the tensor-core prefill path (at most 256)
};

struct LayerPtrs {
    const void *qkvQs, *qkvSc;   // [(nHeads+2nKvHeads)*hd][dim]
    const void *woQs, *woSc;     // [dim][nHeads*hd]
    const void *w13Qs, *w13Sc;   // [2*ff][dim] (gate/up interleaved); MoE: [nExperts][2*ff][dim]
    const void *w2Qs, *w2Sc;     // [dim][ff];                          MoE: [nExperts][dim][ff]
    const float *norm0, *norm1, *qNorm, *kNorm;
    const float *moeGate;        // [nExperts][dim] f32
};

struct GlobalPtrs {
    const float *embedding;      // [vocabFull][dim] (replicated) or this rank's shard when embRowsPerRank != 0
    const float *embeddingPeers[kApiMaxRanks];   // vocabulary shards of all ranks (peer-mapped), used when embRowsPerRank != 0
    uint32_t embRowsPerRank;     // 0: `embedding` is the whole table
    const float *finalNorm;
    const void *wclsQs, *wclsSc; // [vocab][dim]
    const float *rope;           // [seqLen][hd/2][2]
};

// Device memory owned by the engine (allocated and zeroed by dl_engine_create) that a front end reads or writes.
struct EngineBuffers {
    int *tokens, *pos;           // [maxBatch] tokens and positions of a forward; decoding advances tokens[0] / pos[0] on the device
    int *history;                // [seqLen + 1] generated token per position
    float *logits;               // [maxBatch][vocab]
    float *x;                    // [maxBatch][dim] residual stream
    int *pTokens, *pPos;         // [maxPrefill] tokens and positions of a prefill chunk
    void *const *kCache, *const *vCache;   // [nLayers] (host arrays) bf16 [nKvHeads][seqLen][hd]
    int *pTargets;               // [maxPrefill] dl_engine_score: target of each row (global id, -1 = none)
    float *pLogprob;             // [maxPrefill] dl_engine_score results: log P(target), NaN without a target
    int *pTopId;                 //              top-1 id (ids >= the vocabulary limit excluded, lowest index on ties)
    float *pTopLogprob;          //              its log-probability
};

struct CommPtrs {   // mirrored by ctypes
    void *arena[kApiMaxRanks];          // every rank's symmetric arena (dl_engine_arena_bytes each) mapped into this process
    void *mcArena;                      // NVLS multicast mapping of the arena (null: none)
};

}  // namespace dl

extern "C" {
void *dl_engine_create(const dl::EngineConfig *cfg);   // allocates on the current device; null on failure
void dl_engine_destroy(void *h);
int dl_engine_set_layer(void *h, uint32_t layer, const dl::LayerPtrs *p);
int dl_engine_set_globals(void *h, const dl::GlobalPtrs *p);
int dl_engine_get_config(void *h, dl::EngineConfig *cfg);   // the values the engine uses (defaults and limits applied)
int dl_engine_buffers(void *h, dl::EngineBuffers *b);
size_t dl_engine_arena_bytes(const dl::EngineConfig *cfg);   // peer arena per rank for tensor parallelism; no CUDA calls
int dl_engine_set_comm(void *h, const dl::CommPtrs *p);
int dl_engine_enable_mega(void *h, int enable);
int dl_engine_set_vocab_limit(void *h, uint32_t limit);   // greedy arg-max never returns ids >= limit (tokenizer vocabulary size)
int dl_engine_aborted(void *h);
int dl_engine_mega_active(void *h);   // 1 if the last single-token forward ran on the persistent kernel (0: fell back to the multi-kernel path)
unsigned long long dl_engine_sync_ns(void *h);
int dl_engine_sampler_seed(void *h, unsigned long long seed);
int dl_engine_sample(void *h, float temperature, float topp, cudaStream_t stream);   // after a forward with logitsMode 1
int dl_engine_set_trace(void *h, uint64_t *buf, uint32_t capLaunches);
int dl_engine_set_trace_all(void *h, int allCtas);
int dl_engine_forward(void *h, int nb, int logitsMode, int greedyAdvance, cudaStream_t stream);
int dl_engine_forward_part(void *h, int nb, uint32_t layer, int part, float *ybuf, cudaStream_t stream);
int dl_engine_prefill(void *h, uint32_t T, uint32_t p0, int wantLogits, cudaStream_t stream);   // T tokens staged in pTokens/pPos at positions p0 .. p0 + T - 1
// Scores T tokens staged in pTokens/pPos/pTargets at positions p0 .. p0 + T - 1: the prefill chain (same KV rows as dl_engine_prefill),
// the logits of every token, then log-probabilities over the whole vocabulary into pLogprob/pTopId/pTopLogprob. Every rank of a
// tensor-parallel job gets bit-identical results. T <= dl_engine_score_max_tokens; -35 for dense weight files.
int dl_engine_score(void *h, uint32_t T, uint32_t p0, cudaStream_t stream);
uint32_t dl_engine_score_max_tokens(void *h);
int dl_engine_capture_decode(void *h);
int dl_engine_decode_graph(void *h, int nSteps, cudaStream_t stream);
// symmetric peer-memory arena (csrc/cuda/comm_vmm.cu): create (local, binds the bootstrap socket) -> [job-wide barrier] -> connect
// (collective: exchanges file descriptors, maps every peer, sets up the NVSwitch multicast mapping)
void *dl_vmm_create(uint32_t rank, uint32_t nRanks, size_t bytes, const char *tag, int wantMulticast);
int dl_vmm_connect(void *h);
void *dl_vmm_ptr(void *h, uint32_t rank);
void *dl_vmm_mc_ptr(void *h);
int dl_vmm_barrier(void *h, uint32_t phase);   // host barrier over the bootstrap sockets, phase 3..14
void dl_vmm_destroy(void *h);
int dl_repack_q40(const void *src, uint64_t srcRowPitch, uint64_t srcColByteOffset, uint32_t rows, uint32_t blocksPerRow, void *dstQs,
                  void *dstScales, uint32_t dstRowStride, uint32_t dstRowOffset, uint32_t headDim, cudaStream_t stream);
}
