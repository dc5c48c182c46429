#include "native_engine.hpp"

#include <cuda_runtime.h>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <cstring>
#include <map>
#include <stdexcept>
#include <tuple>

#include "../cuda/engine_api.h"

namespace dl {

namespace {

void cudaCheck(cudaError_t e, const char *what) {
    if (e != cudaSuccess) throw std::runtime_error(std::string(what) + ": " + cudaGetErrorString(e));
}
void engCheck(int rc, const char *what) {
    if (rc != 0) throw std::runtime_error(std::string(what) + " failed with code " + std::to_string(rc));
}

struct Mapping {   // read-only mmap of the model file
    const uint8_t *data = nullptr;
    size_t size = 0;
    explicit Mapping(const std::string &path) {
        const int fd = ::open(path.c_str(), O_RDONLY);
        if (fd < 0) throw std::runtime_error("Cannot open model file: " + path);
        struct stat st {};
        if (::fstat(fd, &st) != 0) { ::close(fd); throw std::runtime_error("Cannot stat model file: " + path); }
        size = (size_t)st.st_size;
        void *p = ::mmap(nullptr, size, PROT_READ, MAP_PRIVATE, fd, 0);
        ::close(fd);
        if (p == MAP_FAILED) throw std::runtime_error("Cannot mmap model file: " + path);
        data = (const uint8_t *)p;
    }
    ~Mapping() { if (data) ::munmap((void *)data, size); }
};

struct Q40Dev {   // device layout of csrc/cuda/common.cuh: qs u32 [rows][n/8], scales f16 [rows][n/32]
    void *qs = nullptr, *scales = nullptr;
};

}  // namespace

struct NativeEngine::Impl {
    std::vector<void *> allocations;
    void *engine = nullptr;
    void *vmm = nullptr;               // peer-memory arena handle (tensor parallel)
    cudaStream_t stream = nullptr;
    // weights
    float *embedding = nullptr, *finalNorm = nullptr, *rope = nullptr;
    Q40Dev wcls;
    struct Layer {
        Q40Dev qkv, wo, w13, w2;
        float *norm0 = nullptr, *norm1 = nullptr, *qNorm = nullptr, *kNorm = nullptr, *moeGate = nullptr;
    };
    std::vector<Layer> layers;
    EngineBuffers buf{};   // engine-owned inputs / outputs
    std::vector<float> hostLogits;
    std::map<std::tuple<std::string, uint32_t, uint32_t>, const TensorEntry *> index;
    const TensorEntry &entry(const std::string &name, uint32_t layer = 0, uint32_t expert = 0) const {
        auto it = index.find(std::make_tuple(name, layer, expert));
        if (it == index.end()) throw std::runtime_error("tensor not found in the model file: " + name);
        return *it->second;
    }
};

void *NativeEngine::dev(size_t bytes) {
    void *p = nullptr;
    if (bytes == 0) bytes = 16;
    cudaCheck(cudaMalloc(&p, bytes), "cudaMalloc");
    impl_->allocations.push_back(p);
    cudaCheck(cudaMemsetAsync(p, 0, bytes, impl_->stream), "cudaMemset");   // every later write to p is ordered on the same stream
    return p;
}

NativeEngine::NativeEngine(const std::string &modelPath, uint32_t maxSeqLen, int device, uint32_t rank, uint32_t nRanks,
                           const std::string &commTag, std::function<void()> hostBarrier) {
    rank_ = rank; nRanks_ = std::max(1u, nRanks);
    h_ = loadModelHeader(modelPath, maxSeqLen);
    if (h_.weightType != F_Q40)
        throw std::runtime_error("dllama-native runs q40 weight files; f32/f16/q80 files are served by the Python front end (./dllama)");
    if (h_.headDim != 64 && h_.headDim != 128) throw std::runtime_error("unsupported head dimension");
    dir_ = buildTensorDirectory(h_, true);
    seqLen_ = h_.seqLen;
    impl_ = new Impl();
    try {
        cudaCheck(cudaSetDevice(device), "cudaSetDevice");
        cudaCheck(cudaStreamCreateWithFlags(&impl_->stream, cudaStreamNonBlocking), "cudaStreamCreate");
        for (const TensorEntry &t : dir_) impl_->index[std::make_tuple(t.name, t.layer, t.expert)] = &t;
        const uint32_t hd = h_.headDim, dim = h_.dim, vocab = h_.vocabSize, N = nRanks_;
        // tensor-parallel placement (same rules as distributed_llama_b200/models/loader.py; reference slicers src/nn/nn-core.cpp:223-322):
        // more ranks than KV heads -> nRanks / nKvHeads ranks share one KV head, each with its own query heads of that group
        uint32_t kvRep = 1;
        if (N > h_.nKvHeads) {
            if (N % h_.nKvHeads || (h_.nHeads / h_.nKvHeads) % (N / h_.nKvHeads))
                throw std::runtime_error("the number of GPUs must be a multiple of nKvHeads that divides the query heads of a KV group");
            kvRep = N / h_.nKvHeads;
        }
        if (h_.nHeads % N || (kvRep == 1 && h_.nKvHeads % N) || h_.ffDim() % N || vocab % N)
            throw std::runtime_error("nHeads, nKvHeads, ffDim and vocabSize must be divisible by the number of GPUs");
        headsL_ = h_.nHeads / N; kvHeadsL_ = kvRep > 1 ? 1 : h_.nKvHeads / N;
        kvRank_ = rank_ / kvRep; kvSlices_ = N / kvRep;
        ffL_ = h_.ffDim() / N; vocabL_ = vocab / N;
        const uint32_t ff = ffL_;
        const uint32_t qDim = headsL_ * hd, kvDim = kvHeadsL_ * hd;
        if (N > 1 && (qDim % 128 || ff % 128))
            throw std::runtime_error("per-GPU slices of WO / W2 must be multiples of 128 columns (use fewer GPUs)");
        qkvDim_ = qDim + 2 * kvDim;

        Mapping file(modelPath);
        uploadWeights(file.data);

        Impl &I = *impl_;
        I.hostLogits.resize(vocab);
        EngineConfig cfg{};
        cfg.dim = dim; cfg.nLayers = h_.nLayers; cfg.nHeads = headsL_; cfg.nKvHeads = kvHeadsL_; cfg.headDim = hd; cfg.ffDim = ff;
        cfg.vocab = vocabL_; cfg.seqLen = seqLen_; cfg.nExperts = h_.nExperts; cfg.nActiveExperts = h_.nActiveExperts; cfg.maxBatch = maxBatch_;
        cfg.rank = rank_; cfg.nRanks = N; cfg.eps = h_.normEpsilon; cfg.usePdl = 1;
        cfg.moeFirstExpert = 0; cfg.moeNumLocal = h_.nExperts; cfg.wType = 0;
        cfg.hiddenAct = h_.hiddenAct == ACT_GELU ? 1u : 0u;
        cfg.vocabFull = vocab; cfg.maxPrefill = maxPrefill_;
        I.engine = dl_engine_create(&cfg);
        if (!I.engine) throw std::runtime_error("dl_engine_create failed");
        engCheck(dl_engine_get_config(I.engine, &cfg), "dl_engine_get_config");
        maxBatch_ = cfg.maxBatch; maxPrefill_ = cfg.maxPrefill;
        engCheck(dl_engine_buffers(I.engine, &I.buf), "dl_engine_buffers");
        for (uint32_t l = 0; l < h_.nLayers; l++) {
            const Impl::Layer &L = I.layers[l];
            LayerPtrs lp{};
            lp.qkvQs = L.qkv.qs; lp.qkvSc = L.qkv.scales; lp.woQs = L.wo.qs; lp.woSc = L.wo.scales;
            lp.w13Qs = L.w13.qs; lp.w13Sc = L.w13.scales; lp.w2Qs = L.w2.qs; lp.w2Sc = L.w2.scales;
            lp.norm0 = L.norm0; lp.norm1 = L.norm1; lp.qNorm = L.qNorm; lp.kNorm = L.kNorm; lp.moeGate = L.moeGate;
            engCheck(dl_engine_set_layer(I.engine, l, &lp), "dl_engine_set_layer");
        }
        GlobalPtrs g{};
        g.embedding = I.embedding; g.finalNorm = I.finalNorm; g.wclsQs = I.wcls.qs; g.wclsSc = I.wcls.scales; g.rope = I.rope;
        engCheck(dl_engine_set_globals(I.engine, &g), "dl_engine_set_globals");
        if (N > 1) {
            const size_t bytes = dl_engine_arena_bytes(&cfg);   // symmetric peer-memory arena
            I.vmm = dl_vmm_create(rank_, N, bytes, commTag.c_str(), 1);
            if (!I.vmm) throw std::runtime_error("cannot create the peer-memory arena (CUDA VMM with POSIX file-descriptor handles is required)");
            if (hostBarrier) hostBarrier();      // every rank has bound its bootstrap socket
            engCheck(dl_vmm_connect(I.vmm), "dl_vmm_connect");
            cudaCheck(cudaMemsetAsync(dl_vmm_ptr(I.vmm, rank_), 0, bytes, I.stream), "cudaMemset(arena)");
            cudaCheck(cudaStreamSynchronize(I.stream), "cudaMemset(arena)");
            engCheck(dl_vmm_barrier(I.vmm, 3), "dl_vmm_barrier");   // nobody pushes into an arena that is still being cleared
            CommPtrs cp{};
            for (uint32_t r = 0; r < N; r++) cp.arena[r] = dl_vmm_ptr(I.vmm, r);
            cp.mcArena = dl_vmm_mc_ptr(I.vmm);
            multicast_ = cp.mcArena != nullptr;
            engCheck(dl_engine_set_comm(I.engine, &cp), "dl_engine_set_comm");
        }
        if (h_.nExperts == 0) {
            engCheck(dl_engine_enable_mega(I.engine, 1), "dl_engine_enable_mega");   // falls back per call if the shape is unsupported
            mega_ = true;
        }
        cudaCheck(cudaDeviceSynchronize(), "weight upload");
    } catch (...) {
        release();
        throw;
    }
}

void NativeEngine::release() {
    if (!impl_) return;
    cudaDeviceSynchronize();
    if (impl_->engine) dl_engine_destroy(impl_->engine);
    if (impl_->vmm) dl_vmm_destroy(impl_->vmm);
    for (void *p : impl_->allocations) cudaFree(p);
    if (impl_->stream) cudaStreamDestroy(impl_->stream);
    delete impl_;
    impl_ = nullptr;
}

NativeEngine::~NativeEngine() { release(); }

// Same device-side fusions as distributed_llama_b200/models/loader.py: q|k|v rows concatenated, w1/w3 rows interleaved,
// NeoX (Qwen3) rotary layout re-ordered to adjacent pairs by the repack kernel, q_norm/k_norm permuted alike.
void NativeEngine::uploadWeights(const uint8_t *file) {
    Impl &I = *impl_;
    const uint32_t hd = h_.headDim, dim = h_.dim, ff = ffL_, vocab = vocabL_;
    const uint32_t qDim = headsL_ * hd, kvDim = kvHeadsL_ * hd;
    const bool neox = h_.ropeType == ROPE_FALCON;
    const uint32_t nExp = std::max(1u, h_.nExperts);
    cudaStream_t st = I.stream;

    uint64_t maxRaw = 0;
    for (const TensorEntry &t : dir_) if (t.type == F_Q40) maxRaw = std::max(maxRaw, t.nBytes);
    void *staging = nullptr;
    cudaCheck(cudaMalloc(&staging, maxRaw + 16), "cudaMalloc(staging)");
    auto q40Alloc = [&](uint64_t rows, uint64_t n) {
        Q40Dev w;
        w.qs = dev(rows * (n / 8) * 4);
        w.scales = dev(rows * (n / 32) * 2);
        return w;
    };
    // rows [slice * rowsLocal, (slice + 1) * rowsLocal) of a file tensor: one contiguous byte range (the reference's row split)
    auto repackRows = [&](const TensorEntry &t, const Q40Dev &dst, uint32_t dstStride, uint32_t dstOff, uint32_t headDim, uint32_t rowsLocal,
                          uint32_t slice) {
        const uint64_t rowBytes = (t.n / 32) * 18, bytes = rowBytes * rowsLocal;
        cudaCheck(cudaMemcpyAsync(staging, file + t.offset + (uint64_t)slice * bytes, bytes, cudaMemcpyHostToDevice, st), "cudaMemcpy(weights)");
        engCheck(dl_repack_q40(staging, rowBytes, 0, rowsLocal, (uint32_t)(t.n / 32), dst.qs, dst.scales, dstStride, dstOff, headDim, st), "dl_repack_q40");
        cudaCheck(cudaStreamSynchronize(st), "repack");   // the staging buffer is re-used by the next tensor
        bytesUploaded_ += bytes;
    };
    // columns [slice * colsLocal, (slice + 1) * colsLocal) of every row (the reference's column split, src/nn/nn-core.cpp:307-322):
    // the rank's 18-byte blocks are gathered on the host so that only its bytes cross PCIe
    std::vector<uint8_t> gather;
    auto repackCols = [&](const TensorEntry &t, const Q40Dev &dst, uint32_t dstOff, uint32_t colsLocal, uint32_t slice) {
        const uint64_t rowBytes = (t.n / 32) * 18, locBytes = (uint64_t)(colsLocal / 32) * 18;
        const uint8_t *src = file + t.offset;
        if (locBytes != rowBytes) {
            gather.resize((size_t)t.d * locBytes);
            for (uint64_t r = 0; r < t.d; r++) std::memcpy(gather.data() + r * locBytes, file + t.offset + r * rowBytes + (uint64_t)slice * locBytes, locBytes);
            src = gather.data();
        }
        cudaCheck(cudaMemcpyAsync(staging, src, (size_t)t.d * locBytes, cudaMemcpyHostToDevice, st), "cudaMemcpy(weights)");
        engCheck(dl_repack_q40(staging, locBytes, 0, (uint32_t)t.d, colsLocal / 32, dst.qs, dst.scales, 1, dstOff, 0, st), "dl_repack_q40");
        cudaCheck(cudaStreamSynchronize(st), "repack");
        bytesUploaded_ += (uint64_t)t.d * locBytes;
    };
    auto f32Tensor = [&](const TensorEntry &t, const std::vector<uint32_t> *perm = nullptr) {
        const size_t count = (size_t)t.d * t.n;
        float *p = (float *)dev(count * 4);
        if (perm) {
            std::vector<float> tmp(count);
            const float *src = (const float *)(file + t.offset);
            for (size_t i = 0; i < count; i++) tmp[i] = src[(*perm)[i]];
            cudaCheck(cudaMemcpyAsync(p, tmp.data(), count * 4, cudaMemcpyHostToDevice, st), "cudaMemcpy(f32)");
            cudaCheck(cudaStreamSynchronize(st), "cudaMemcpy(f32)");
        } else {
            cudaCheck(cudaMemcpyAsync(p, file + t.offset, count * 4, cudaMemcpyHostToDevice, st), "cudaMemcpy(f32)");
        }
        bytesUploaded_ += count * 4;
        return p;
    };
    std::vector<uint32_t> perm(hd);   // new[2j] = old[j], new[2j+1] = old[j + hd/2]
    for (uint32_t j = 0; j < hd / 2; j++) { perm[2 * j] = j; perm[2 * j + 1] = j + hd / 2; }

    I.embedding = f32Tensor(I.entry("embedding"));
    I.finalNorm = f32Tensor(I.entry("final_norm"));
    I.wcls = q40Alloc(vocab, dim);
    repackRows(I.entry("final_matmul_logits"), I.wcls, 1, 0, 0, vocab, rank_);
    {
        std::vector<float> table((size_t)seqLen_ * hd);
        buildRopeTable(h_, seqLen_, table.data());
        I.rope = (float *)dev(table.size() * 4);
        cudaCheck(cudaMemcpyAsync(I.rope, table.data(), table.size() * 4, cudaMemcpyHostToDevice, st), "cudaMemcpy(rope)");
        cudaCheck(cudaStreamSynchronize(st), "cudaMemcpy(rope)");
    }
    I.layers.resize(h_.nLayers);
    for (uint32_t l = 0; l < h_.nLayers; l++) {
        Impl::Layer &L = I.layers[l];
        L.qkv = q40Alloc(qkvDim_, dim);
        repackRows(I.entry("block_matmul_q", l), L.qkv, 1, 0, neox ? hd : 0, qDim, rank_);
        repackRows(I.entry("block_matmul_k", l), L.qkv, 1, qDim, neox ? hd : 0, kvDim, kvRank_);
        repackRows(I.entry("block_matmul_v", l), L.qkv, 1, qDim + kvDim, 0, kvDim, kvRank_);
        L.wo = q40Alloc(dim, qDim);
        repackCols(I.entry("block_matmul_wo", l), L.wo, 0, qDim, rank_);
        L.w13 = q40Alloc((uint64_t)nExp * 2 * ff, dim);
        L.w2 = q40Alloc((uint64_t)nExp * dim, ff);
        for (uint32_t e = 0; e < nExp; e++) {
            repackRows(I.entry("block_matmul_w1", l, e), L.w13, 2, e * 2 * ff, 0, ff, rank_);
            repackRows(I.entry("block_matmul_w3", l, e), L.w13, 2, e * 2 * ff + 1, 0, ff, rank_);
            repackCols(I.entry("block_matmul_w2", l, e), L.w2, e * dim, ff, rank_);
        }
        L.norm0 = f32Tensor(I.entry("block_norm_0", l));
        L.norm1 = f32Tensor(I.entry("block_norm_1", l));
        if (h_.qkNorm()) {
            L.qNorm = f32Tensor(I.entry("block_norm_q", l), neox ? &perm : nullptr);
            L.kNorm = f32Tensor(I.entry("block_norm_k", l), neox ? &perm : nullptr);
        }
        if (h_.nExperts > 0) L.moeGate = f32Tensor(I.entry("block_moe_gate", l));
    }
    cudaCheck(cudaStreamSynchronize(st), "weight upload");
    cudaFree(staging);
}

void NativeEngine::setInputs(const int32_t *tokens, uint32_t n, uint32_t pos, bool prefillBuffers) {
    std::vector<int32_t> p(n);
    for (uint32_t i = 0; i < n; i++) p[i] = (int32_t)(pos + i);
    Impl &I = *impl_;
    // pageable sources: the copies are staged before the call returns, so the vectors may die right away
    cudaCheck(cudaMemcpyAsync(prefillBuffers ? I.buf.pTokens : I.buf.tokens, tokens, n * 4, cudaMemcpyHostToDevice, I.stream), "cudaMemcpy(tokens)");
    cudaCheck(cudaMemcpyAsync(prefillBuffers ? I.buf.pPos : I.buf.pos, p.data(), n * 4, cudaMemcpyHostToDevice, I.stream), "cudaMemcpy(pos)");
}

void NativeEngine::forward(uint32_t n, int logitsMode, bool greedyAdvance) {
    engCheck(dl_engine_forward(impl_->engine, (int)n, logitsMode, greedyAdvance ? 1 : 0, impl_->stream), "dl_engine_forward");
}

void NativeEngine::prefill(const std::vector<int32_t> &tokens, uint32_t pos) {
    if (pos + tokens.size() > seqLen_) throw std::runtime_error("position beyond the context length");
    const bool tc = h_.nExperts == 0 || (h_.dim % 256 == 0 && ffL_ % 256 == 0);   // MoE: grouped tensor-core GEMMs need 256-wide K
    size_t i = 0;
    while (i < tokens.size()) {
        const size_t rem = tokens.size() - i;
        uint32_t n;
        if (tc && rem >= 9) {
            n = (uint32_t)std::min<size_t>(rem, maxPrefill_);
            setInputs(tokens.data() + i, n, pos + (uint32_t)i, true);
            engCheck(dl_engine_prefill(impl_->engine, n, pos + (uint32_t)i, 0, impl_->stream), "dl_engine_prefill");
        } else {
            n = 1;
            while (n * 2 <= std::min<size_t>(rem, maxBatch_)) n *= 2;
            setInputs(tokens.data() + i, n, pos + (uint32_t)i, false);
            forward(n, 0, false);
        }
        i += n;
    }
}

const float *NativeEngine::step(int32_t token, uint32_t pos) {
    if (nRanks_ > 1) throw std::runtime_error("host-side logits are not gathered under tensor parallelism: use stepGreedy / stepSampled");
    if (pos >= seqLen_) throw std::runtime_error("position beyond the context length");
    setInputs(&token, 1, pos, false);
    forward(1, 1, false);
    Impl &I = *impl_;
    cudaCheck(cudaMemcpyAsync(I.hostLogits.data(), I.buf.logits, (size_t)h_.vocabSize * 4, cudaMemcpyDeviceToHost, I.stream), "cudaMemcpy(logits)");
    cudaCheck(cudaStreamSynchronize(I.stream), "step");
    return I.hostLogits.data();
}

std::vector<int32_t> NativeEngine::decodeGreedy(int32_t firstToken, uint32_t pos, uint32_t nSteps) {
    if (pos + nSteps > seqLen_) throw std::runtime_error("decode would run past the context length");
    Impl &I = *impl_;
    setInputs(&firstToken, 1, pos, false);
    if (!graphReady_) {
        // warm-up run configures kernel attributes outside of capture; inputs are restored afterwards
        forward(1, 1, false);
        cudaCheck(cudaStreamSynchronize(I.stream), "warm-up");
        engCheck(dl_engine_capture_decode(I.engine), "dl_engine_capture_decode");
        graphReady_ = true;
        setInputs(&firstToken, 1, pos, false);
    }
    engCheck(dl_engine_decode_graph(I.engine, (int)nSteps, I.stream), "dl_engine_decode_graph");
    std::vector<int32_t> out(nSteps);
    cudaCheck(cudaMemcpyAsync(out.data(), I.buf.history + pos + 1, (size_t)nSteps * 4, cudaMemcpyDeviceToHost, I.stream), "cudaMemcpy(history)");
    cudaCheck(cudaStreamSynchronize(I.stream), "decode");
    return out;
}

int32_t NativeEngine::stepGreedy(int32_t token, uint32_t pos) {
    if (pos >= seqLen_) throw std::runtime_error("position beyond the context length");
    Impl &I = *impl_;
    setInputs(&token, 1, pos, false);
    if (!graphReady_) {
        forward(1, 1, false);
        cudaCheck(cudaStreamSynchronize(I.stream), "warm-up");
        engCheck(dl_engine_capture_decode(I.engine), "dl_engine_capture_decode");
        graphReady_ = true;
        setInputs(&token, 1, pos, false);
    }
    engCheck(dl_engine_decode_graph(I.engine, 1, I.stream), "dl_engine_decode_graph");
    int32_t next = 0;   // the arg-max kernel leaves the sampled token in tokens[0] (and advances pos[0]) on the device
    cudaCheck(cudaMemcpyAsync(&next, I.buf.tokens, 4, cudaMemcpyDeviceToHost, I.stream), "cudaMemcpy(token)");
    cudaCheck(cudaStreamSynchronize(I.stream), "stepGreedy");
    if (nRanks_ > 1 && dl_engine_aborted(I.engine)) throw std::runtime_error("device-side wait timed out: a tensor-parallel peer stopped responding");
    return next;
}

void NativeEngine::seedSampler(uint64_t seed) { engCheck(dl_engine_sampler_seed(impl_->engine, seed), "dl_engine_sampler_seed"); }

int32_t NativeEngine::stepSampled(int32_t token, uint32_t pos, float temperature, float topp) {
    if (pos >= seqLen_) throw std::runtime_error("position beyond the context length");
    Impl &I = *impl_;
    setInputs(&token, 1, pos, false);
    forward(1, 1, false);
    engCheck(dl_engine_sample(I.engine, temperature, topp, I.stream), "dl_engine_sample");
    int32_t next = 0;   // the sampler leaves the drawn token in tokens[0]
    cudaCheck(cudaMemcpyAsync(&next, I.buf.tokens, 4, cudaMemcpyDeviceToHost, I.stream), "cudaMemcpy(token)");
    cudaCheck(cudaStreamSynchronize(I.stream), "stepSampled");
    if (dl_engine_aborted(I.engine)) throw std::runtime_error("device-side wait timed out: a tensor-parallel peer stopped responding");
    return next;
}

uint64_t NativeEngine::syncNs() const { return nRanks_ > 1 ? (uint64_t)dl_engine_sync_ns(impl_->engine) : 0; }

void NativeEngine::linkBytes(uint32_t nTokens, uint64_t &sent, uint64_t &received) const {
    sent = received = 0;
    if (nRanks_ <= 1) return;
    const uint64_t perAr = (uint64_t)nTokens * h_.dim * 8;
    sent = 2ull * h_.nLayers * perAr * (multicast_ ? 1 : nRanks_ - 1);
    received = 2ull * h_.nLayers * perAr * (nRanks_ - 1);
}

void NativeEngine::synchronize() { cudaCheck(cudaStreamSynchronize(impl_->stream), "synchronize"); }

void NativeEngine::setVocabLimit(uint32_t limit) {
    if (limit >= h_.vocabSize) limit = 0;
    engCheck(dl_engine_set_vocab_limit(impl_->engine, limit), "dl_engine_set_vocab_limit");
    graphReady_ = false;   // the limit is a launch parameter of the captured step
}

}  // namespace dl
