// Python-free runtime of one GPU: maps a `.m` file, uploads + re-tiles the q40 weights and drives the
// engine in _cuda.so (persistent decode kernel, tcgen05 prefill, CUDA-graph greedy loop).
//
// Role in the reference: loadLlmNetWeight + NnExecutor/NnCpuDevice set-up + RootLlmInference (src/llm.cpp:614-669,
// src/nn/nn-cpu.cpp:41-148, src/app.cpp:168-208) for the single-node case. The tensor-parallel launcher (one process per GPU,
// torch.distributed bootstrap, peer-memory arena) lives in the Python package; this class is what `dllama-native` and embedders
// that do not want an interpreter link against.
#pragma once
#include <cstdint>
#include <functional>
#include <string>
#include <vector>

#include "../host/model_format.hpp"

namespace dl {

class NativeEngine {
public:
    // maxSeqLen == 0: the model's context length. Throws std::runtime_error on unsupported files / CUDA errors.
    // Tensor parallel (nRanks > 1, one process per GPU of one NVSwitch box): this rank uploads only its slice of every matrix
    // (row slices of q/k/v/w1/w3/logits, column slices of wo/w2 gathered on the host; KV heads are replicated when there are more
    // ranks than KV heads), creates its part of the symmetric peer-memory arena (csrc/cuda/comm_vmm.cu: CUDA VMM + NVSwitch
    // multicast, bootstrapped over unix sockets named after `commTag`) and the kernels do their all-reduces over it. `hostBarrier`
    // must synchronise all ranks of the job (it is called between the two bootstrap steps). Every rank then issues the same
    // sequence of prefill / step calls (reference: root + `dllama worker` processes, src/dllama.cpp:260-285).
    NativeEngine(const std::string &modelPath, uint32_t maxSeqLen, int device, uint32_t rank = 0, uint32_t nRanks = 1,
                 const std::string &commTag = std::string(), std::function<void()> hostBarrier = std::function<void()>());
    ~NativeEngine();
    NativeEngine(const NativeEngine &) = delete;
    NativeEngine &operator=(const NativeEngine &) = delete;

    const ModelHeader &header() const { return h_; }
    uint32_t seqLen() const { return seqLen_; }
    uint64_t bytesUploaded() const { return bytesUploaded_; }
    uint32_t rank() const { return rank_; }
    uint32_t nRanks() const { return nRanks_; }
    bool multicast() const { return multicast_; }
    bool persistentKernel() const { return mega_; }

    // Feeds prompt tokens at positions [pos, pos + n): chunks of up to 192 tokens on the tensor-core path (dense models),
    // power-of-two batches of up to 8 on the GEMV path otherwise. No logits are produced.
    void prefill(const std::vector<int32_t> &tokens, uint32_t pos);
    // One token; returns the logits row (host memory owned by the engine, valid until the next call). Single GPU only: under tensor
    // parallelism the logits stay sharded on the devices (use stepGreedy / stepSampled).
    const float *step(int32_t token, uint32_t pos);
    // One greedy step entirely on the device (graph replay); returns the next token.
    int32_t stepGreedy(int32_t token, uint32_t pos);
    // One step with temperature / top-p sampling on the device (csrc/cuda/sampler.cu; same xorshift* stream as dl::Sampler). Every
    // rank must have called seedSampler with the same seed; under tensor parallelism every rank draws the same token.
    void seedSampler(uint64_t seed);
    int32_t stepSampled(int32_t token, uint32_t pos, float temperature, float topp);
    // n greedy steps back to back on the device without host round trips; returns the generated tokens.
    std::vector<int32_t> decodeGreedy(int32_t firstToken, uint32_t pos, uint32_t nSteps);
    void synchronize();
    // Traffic / synchronisation accounting of the reference's Eval / Pred lines (src/dllama.cpp:59-66): cumulative ns this rank's
    // decode kernel waited for its peers inside the fused all-reduces, and (sent, received) NVLink bytes of a forward over nTokens
    // tokens (2 all-reduces per layer, 8-byte LL words; one multicast store per value when the NVSwitch mapping exists).
    uint64_t syncNs() const;
    void linkBytes(uint32_t nTokens, uint64_t &sent, uint64_t &received) const;
    // Greedy decoding on the device ignores vocabulary rows >= limit (tokenizer vocabulary smaller than the embedding table).
    void setVocabLimit(uint32_t limit);

private:
    struct Impl;
    void *dev(size_t bytes);            // zero-initialised device allocation for weights, owned by the engine
    void release();
    void uploadWeights(const uint8_t *file);
    void setInputs(const int32_t *tokens, uint32_t n, uint32_t pos, bool prefillBuffers);
    void forward(uint32_t n, int logitsMode, bool greedyAdvance);

    ModelHeader h_;
    std::vector<TensorEntry> dir_;
    uint32_t seqLen_ = 0, maxBatch_ = 8, maxPrefill_ = 192, qkvDim_ = 0;
    uint32_t rank_ = 0, nRanks_ = 1, kvRank_ = 0, kvSlices_ = 1;          // tensor-parallel placement of this process
    uint32_t headsL_ = 0, kvHeadsL_ = 0, ffL_ = 0, vocabL_ = 0;          // per-rank slice sizes
    bool mega_ = false, graphReady_ = false, multicast_ = false;
    uint64_t bytesUploaded_ = 0;
    Impl *impl_ = nullptr;
};

}  // namespace dl
