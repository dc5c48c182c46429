"""`.m` file -> device weights of one tensor-parallel rank.

Reference behaviour replaced: loadLlmNetWeight + NnRootWeightLoader (src/llm.cpp:614-669,
src/nn/nn-network.cpp:797-888): the root walks the file, splits every tensor on the CPU and streams the slices
to workers over TCP. Here every rank maps the file, uploads the byte range that contains its rows and lets the
`repack_q40` kernel cut the column slice and re-tile into the device layout on the GPU (see csrc/cuda/repack.cu).
Partition rules are the reference's (row split for q,k,v,w1,w3,wcls; column split for wo,w2; SURVEY A.6).

Device-side fusions prepared here:
  * q|k|v rows concatenated into one matrix  (one GEMV/GEMM per layer instead of three)
  * w1/w3 rows interleaved (gate_i, up_i)     (SwiGLU in the epilogue of one kernel)
  * NeoX/"Falcon" rotary layout (Qwen3) re-ordered to adjacent pairs at load, q_norm/k_norm permuted alike
"""
from __future__ import annotations

import warnings
from dataclasses import dataclass, field
from typing import List, Optional

import numpy as np
import torch

from .. import host
from ..formats.model_file import ModelFile
from ..formats import quants
from ..ops import cuda_lib as cl
from ..ops.q40 import DeviceDense, DeviceQ40, repack_q40
from .config import ROPE_FALCON


@dataclass
class LayerWeights:
    qkv: DeviceQ40
    wo: DeviceQ40
    w13: DeviceQ40
    w2: DeviceQ40
    norm0: torch.Tensor
    norm1: torch.Tensor
    q_norm: Optional[torch.Tensor] = None
    k_norm: Optional[torch.Tensor] = None
    moe_gate: Optional[torch.Tensor] = None


@dataclass
class DeviceWeights:
    header: object
    rank: int
    n_ranks: int
    n_heads: int          # local
    n_kv_heads: int       # local
    ff_dim: int           # local
    vocab: int            # local
    embedding: torch.Tensor
    final_norm: torch.Tensor
    wcls: DeviceQ40
    rope: torch.Tensor
    layers: List[LayerWeights] = field(default_factory=list)
    bytes_uploaded: int = 0
    first_expert: int = 0        # experts held by this rank (expert parallelism), all of them in TP mode
    n_local_experts: int = 0
    moe_mode: str = "tp"
    weight_kind: int = 0         # 0 = q40 device layout, 1 = dense f32, 2 = dense f16
    embedding_ptrs: Optional[List[int]] = None   # vocabulary-sharded embedding: device pointer of every rank's shard (peer mapped)
    embedding_rows: int = 0      # rows per shard (0: `embedding` is the whole replicated table)


def _interleave_perm(head_dim: int) -> np.ndarray:
    """new[2j] = old[j], new[2j+1] = old[j + hd/2]"""
    half = head_dim // 2
    perm = np.empty(head_dim, dtype=np.int64)
    perm[0::2] = np.arange(half)
    perm[1::2] = np.arange(half) + half
    return perm


class _Uploader:
    def __init__(self, mf: ModelFile, device):
        self.mf = mf
        self.device = device
        self.bytes = 0

    def rows(self, entry, first_row: int, n_rows: int) -> torch.Tensor:
        """Uploads full-width rows [first_row, first_row+n_rows) of a tensor as raw bytes."""
        row_bytes = quants.tensor_bytes(entry.type, entry.n)
        off = entry.offset + first_row * row_bytes
        view = self.mf.data[off: off + n_rows * row_bytes]
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            t = torch.from_numpy(view)
        self.bytes += t.numel()
        return t.to(self.device, non_blocking=False)

    def cols(self, entry, first_col_byte: int, n_col_bytes: int) -> torch.Tensor:
        """Uploads the byte columns [first_col_byte, +n_col_bytes) of every row of a tensor: the column slice of one rank is
        gathered on the host (strided view of the mapped file) so only the bytes the rank owns cross PCIe — the reference's
        splitColMatmulWeight does the same cut before streaming a slice to a worker (src/nn/nn-core.cpp:307-322)."""
        row_bytes = quants.tensor_bytes(entry.type, entry.n)
        view = self.mf.data[entry.offset: entry.offset + entry.d * row_bytes].reshape(entry.d, row_bytes)[:, first_col_byte:first_col_byte + n_col_bytes]
        t = torch.from_numpy(np.ascontiguousarray(view))
        self.bytes += t.numel()
        return t.to(self.device, non_blocking=False)

    def f32(self, entry) -> torch.Tensor:
        x = self.mf.tensor_f32(entry)
        self.bytes += x.nbytes
        return torch.from_numpy(np.ascontiguousarray(x)).to(self.device)


def _load_dense(mf: ModelFile, up: "_Uploader", rank, n_ranks, kv_rank, kv_ranks, nh, nkv, ff0, v0, neox, device) -> "DeviceWeights":
    """f32 / f16 / q80 weight files: matrices stay dense on the device (f16 files as f16, everything else as f32 — q80 blocks
    are dequantised exactly) and run through csrc/cuda/gemv_dense.cu with f32 activations. This is the reference's
    F32_F32_F32 matmul path (`--buffer-float-type f32`, src/nn/nn-cpu-ops.cpp:1138-1160); same partition rules."""
    h = mf.header
    H = host()
    hd, dim = h.head_dim, h.dim
    dt = torch.float16 if h.weight_type == quants.F_16 else torch.float32

    def sliced(name, layer, r, n):
        x = mf.slice_f32(mf.entry(name, layer, 0), r, n)
        up.bytes += x.nbytes
        return torch.from_numpy(np.ascontiguousarray(x))

    def heads_interleaved(x, n_heads):
        if not neox:
            return x
        perm = torch.from_numpy(_interleave_perm(hd))
        return x.reshape(n_heads, hd, x.shape[1])[:, perm, :].reshape(n_heads * hd, x.shape[1])

    def dev(x, d, n):
        return DeviceDense(x.to(dt).contiguous().to(device), d, n)

    W = DeviceWeights(header=h, rank=rank, n_ranks=n_ranks, n_heads=nh, n_kv_heads=nkv, ff_dim=ff0, vocab=v0,
                      embedding=up.f32(mf.entry("embedding")), final_norm=up.f32(mf.entry("final_norm")),
                      wcls=dev(sliced("final_matmul_logits", 0, rank, n_ranks), v0, dim),
                      rope=torch.from_numpy(np.asarray(H.build_rope_table(h, h.seq_len))).to(device))
    perm_dev = torch.from_numpy(_interleave_perm(hd)).to(device) if neox else None
    for l in range(h.n_layers):
        q = heads_interleaved(sliced("block_matmul_q", l, rank, n_ranks), nh)
        k = heads_interleaved(sliced("block_matmul_k", l, kv_rank, kv_ranks), nkv)
        v = sliced("block_matmul_v", l, kv_rank, kv_ranks)
        w1, w3 = sliced("block_matmul_w1", l, rank, n_ranks), sliced("block_matmul_w3", l, rank, n_ranks)
        L = LayerWeights(qkv=dev(torch.cat([q, k, v], 0), (nh + 2 * nkv) * hd, dim),
                         wo=dev(sliced("block_matmul_wo", l, rank, n_ranks), dim, nh * hd),
                         w13=dev(torch.stack([w1, w3], 1).reshape(2 * ff0, dim), 2 * ff0, dim),
                         w2=dev(sliced("block_matmul_w2", l, rank, n_ranks), dim, ff0),
                         norm0=up.f32(mf.entry("block_norm_0", l)), norm1=up.f32(mf.entry("block_norm_1", l)))
        if h.qk_norm:
            qn, kn = up.f32(mf.entry("block_norm_q", l)), up.f32(mf.entry("block_norm_k", l))
            L.q_norm = qn[perm_dev].contiguous() if neox else qn
            L.k_norm = kn[perm_dev].contiguous() if neox else kn
        W.layers.append(L)
    if torch.device(device).type == "cuda":
        torch.cuda.synchronize(device)
    W.bytes_uploaded = up.bytes
    W.weight_kind = 1 if dt == torch.float32 else 2
    return W


def _sharded_embedding(mf: ModelFile, up: "_Uploader", rank: int, n_ranks: int, device, comm):
    """Uploads only this rank's vocabulary rows of the f32 embedding into peer-mapped memory; returns (local tensor, pointers of all
    shards, rows per shard) or None when no symmetric allocation is available (the table is then replicated)."""
    import os
    h = mf.header
    if comm is None or n_ranks <= 1 or h.vocab_size % n_ranks or os.environ.get("DL_REPLICATE_EMBEDDING") is not None:
        return None
    if not hasattr(comm, "alloc_shared"):
        return None
    rows = h.vocab_size // n_ranks
    ptrs = comm.alloc_shared(rows * h.dim * 4)
    if ptrs is None:
        return None
    local = cl.device_view(ptrs[rank], (rows, h.dim), torch.float32, device=device)
    e = mf.entry("embedding")
    src = mf.data[e.offset + rank * rows * h.dim * 4: e.offset + (rank + 1) * rows * h.dim * 4]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        host_t = torch.from_numpy(src).view(torch.float32).view(rows, h.dim)
    local.copy_(host_t)
    up.bytes += rows * h.dim * 4
    torch.cuda.synchronize(device)
    import torch.distributed as dist
    dist.barrier()          # every shard is in place before any rank may read a peer's rows
    return local, ptrs, rows


def load_device_weights(mf: ModelFile, rank: int = 0, n_ranks: int = 1, device="cuda", moe_mode: str = "auto", comm=None) -> DeviceWeights:
    """moe_mode (Qwen3-MoE only): "tp" slices every expert over the ranks like the reference (src/llm.cpp:454-486);
    "ep" gives each rank nExperts/nRanks whole experts (expert parallelism: the expert FFN streams full-width matrices and the
    combine is the same in-kernel all-reduce); "auto" picks ep when the TP slice would be narrower than 128 columns."""
    h = mf.header
    dense = h.weight_type != quants.F_Q40
    if dense and h.n_experts > 0:
        raise NotImplementedError("mixture-of-experts models need q40 weights (the expert-routed kernels are q40 only)")
    H = host()
    if moe_mode == "auto":
        moe_mode = "ep" if (h.n_experts > 0 and n_ranks > 1 and (h.ff_dim // n_ranks) % 128 != 0 and h.n_experts % n_ranks == 0) else "tp"
    ep = h.n_experts > 0 and moe_mode == "ep" and n_ranks > 1
    if ep and h.n_experts % n_ranks:
        raise ValueError("nExperts must be divisible by the number of ranks for expert parallelism")
    # KV-head replication: with more ranks than KV heads (the reference refuses this, src/app.cpp:236-238) groups of
    # nRanks/nKvHeads ranks share one KV head; every rank still owns a distinct set of query heads of that group.
    kv_rep = 1
    if n_ranks > h.n_kv_heads:
        if n_ranks % h.n_kv_heads or (h.n_heads // h.n_kv_heads) % (n_ranks // h.n_kv_heads):
            raise ValueError("nRanks must be a multiple of nKvHeads that divides the query heads of a KV group")
        kv_rep = n_ranks // h.n_kv_heads
    if h.n_heads % n_ranks or (kv_rep == 1 and h.n_kv_heads % n_ranks) or (not ep and h.ff_dim % n_ranks) or h.vocab_size % n_ranks:
        raise ValueError("nHeads, nKvHeads, ffDim and vocabSize must be divisible by the number of ranks")
    hd = h.head_dim
    nh, nkv = h.n_heads // n_ranks, (1 if kv_rep > 1 else h.n_kv_heads // n_ranks)
    kv_rank = rank // kv_rep       # which KV slice this rank reads
    kv_ranks = n_ranks // kv_rep   # number of distinct KV slices
    q0, kv0, ff0, v0 = nh * hd, nkv * hd, (h.ff_dim if ep else h.ff_dim // n_ranks), h.vocab_size // n_ranks
    if (q0 % 32) or (ff0 % 32):
        raise ValueError("column slices must cover whole 32-element quant blocks")
    neox = h.rope_type == ROPE_FALCON
    up = _Uploader(mf, device)
    dim = h.dim
    if dense:
        return _load_dense(mf, up, rank, n_ranks, kv_rank, kv_ranks, nh, nkv, ff0, v0, neox, device)

    def row_sliced(name, layer, expert, dst: DeviceQ40, rows_local, dst_stride=1, dst_off=0, head_dim=0, slice_rank=None):
        e = mf.entry(name, layer, expert)
        raw = up.rows(e, (rank if slice_rank is None else slice_rank) * rows_local, rows_local)
        repack_q40(raw, rows_local, e.n, dst, dst_row_stride=dst_stride, dst_row_offset=dst_off, head_dim=head_dim)

    def col_sliced(name, layer, expert, dst: DeviceQ40, cols_local, dst_off=0, slice_rank=None):
        e = mf.entry(name, layer, expert)
        cbytes = quants.tensor_bytes(e.type, cols_local)
        if cbytes == quants.tensor_bytes(e.type, e.n):
            raw = up.rows(e, 0, e.d)
        else:
            raw = up.cols(e, (rank if slice_rank is None else slice_rank) * cbytes, cbytes)
        repack_q40(raw, e.d, cols_local, dst, src_row_pitch=cbytes, src_col_byte_offset=0, dst_row_offset=dst_off)

    shard = _sharded_embedding(mf, up, rank, n_ranks, device, comm)
    W = DeviceWeights(header=h, rank=rank, n_ranks=n_ranks, n_heads=nh, n_kv_heads=nkv, ff_dim=ff0, vocab=v0,
                      embedding=shard[0] if shard else up.f32(mf.entry("embedding")), final_norm=up.f32(mf.entry("final_norm")),
                      wcls=DeviceQ40.empty(v0, dim, device),
                      rope=torch.from_numpy(np.asarray(H.build_rope_table(h, h.seq_len))).to(device))
    if shard:
        W.embedding_ptrs, W.embedding_rows = shard[1], shard[2]
    row_sliced("final_matmul_logits", 0, 0, W.wcls, v0)
    perm = torch.from_numpy(_interleave_perm(hd)).to(device) if neox else None
    n_exp = max(h.n_experts, 1)
    first_exp, n_local = (rank * (h.n_experts // n_ranks), h.n_experts // n_ranks) if ep else (0, n_exp)
    W.first_expert, W.n_local_experts, W.moe_mode = first_exp, (n_local if h.n_experts > 0 else 0), ("ep" if ep else "tp")
    esr = 0 if ep else None      # expert tensors: whole matrices under EP
    for l in range(h.n_layers):
        qkv = DeviceQ40.empty(q0 + 2 * kv0, dim, device)
        row_sliced("block_matmul_q", l, 0, qkv, q0, head_dim=hd if neox else 0)
        row_sliced("block_matmul_k", l, 0, qkv, kv0, dst_off=q0, head_dim=hd if neox else 0, slice_rank=kv_rank)
        row_sliced("block_matmul_v", l, 0, qkv, kv0, dst_off=q0 + kv0, slice_rank=kv_rank)
        wo = DeviceQ40.empty(dim, q0, device)
        col_sliced("block_matmul_wo", l, 0, wo, q0)
        w13 = DeviceQ40.empty(2 * ff0, dim, device, lead=n_local)
        w2 = DeviceQ40.empty(dim, ff0, device, lead=n_local)
        for le in range(n_local):
            e = first_exp + le
            row_sliced("block_matmul_w1", l, e, w13, ff0, dst_stride=2, dst_off=le * 2 * ff0, slice_rank=esr)
            row_sliced("block_matmul_w3", l, e, w13, ff0, dst_stride=2, dst_off=le * 2 * ff0 + 1, slice_rank=esr)
            col_sliced("block_matmul_w2", l, e, w2, ff0, dst_off=le * dim, slice_rank=esr)
        L = LayerWeights(qkv=qkv, wo=wo, w13=w13, w2=w2, norm0=up.f32(mf.entry("block_norm_0", l)),
                         norm1=up.f32(mf.entry("block_norm_1", l)))
        if h.qk_norm:
            qn, kn = up.f32(mf.entry("block_norm_q", l)), up.f32(mf.entry("block_norm_k", l))
            L.q_norm = qn[perm].contiguous() if neox else qn
            L.k_norm = kn[perm].contiguous() if neox else kn
        if h.n_experts > 0:
            L.moe_gate = up.f32(mf.entry("block_moe_gate", l))
        W.layers.append(L)
    torch.cuda.synchronize(device)
    W.bytes_uploaded = up.bytes
    return W


def synthetic_device_weights(cfg, rank: int = 0, n_ranks: int = 1, device="cuda", moe_mode: str = "auto", seed: int = 1234,
                             max_seq_len: int = 0) -> DeviceWeights:
    """Random-init weights of architecture `cfg`, created directly in the device layout of this rank (no `.m` file, no upload):
    used to benchmark the large configurations (Qwen3-14B, Qwen3-30B-A3B, Llama-3.3-70B) whose 11-40 GB files would take minutes
    to write on a fresh box. Shapes, partitioning (row / column slices, KV-head replication, expert placement) and value
    statistics follow load_device_weights / write_synthetic_model; the values themselves are not those of a file with that seed."""
    import io
    from ..formats.model_file import write_model_header
    from .config import ARCH_QWEN3, ARCH_QWEN3_MOE
    H = host()
    buf = io.BytesIO()
    write_model_header(buf, cfg.header_params(quants.F_Q40))
    h = H.parse_model_header(buf.getvalue(), 1 << 50, max_seq_len)
    if moe_mode == "auto":
        moe_mode = "ep" if (h.n_experts > 0 and n_ranks > 1 and (h.ff_dim // n_ranks) % 256 != 0 and h.n_experts % n_ranks == 0) else "tp"
    ep = h.n_experts > 0 and moe_mode == "ep" and n_ranks > 1
    kv_rep = 1
    if n_ranks > h.n_kv_heads:
        if n_ranks % h.n_kv_heads or (h.n_heads // h.n_kv_heads) % (n_ranks // h.n_kv_heads):
            raise ValueError("nRanks must be a multiple of nKvHeads that divides the query heads of a KV group")
        kv_rep = n_ranks // h.n_kv_heads
    hd, dim = h.head_dim, h.dim
    nh, nkv = h.n_heads // n_ranks, (1 if kv_rep > 1 else h.n_kv_heads // n_ranks)
    q0, kv0 = nh * hd, nkv * hd
    ff0 = h.ff_dim if ep else h.ff_dim // n_ranks
    v0 = h.vocab_size // n_ranks
    g = torch.Generator(device=device)
    g.manual_seed(seed + 7919 * rank)

    def q40(d, n, std, lead=1):
        w = DeviceQ40.empty(d, n, device, lead=lead)
        w.qs.random_(-2 ** 31, 2 ** 31 - 1, generator=g)
        w.scales.copy_(((std / 4.61) * (0.7 + 0.6 * torch.rand(w.scales.shape, device=device, generator=g))).half())
        return w

    def norm(n):
        return (1.0 + 0.1 * torch.randn(n, device=device, generator=g)).float()

    ge = torch.Generator(device=device)
    ge.manual_seed(seed)      # the embedding is replicated: same values on every rank
    emb = torch.randn(h.vocab_size, dim, device=device, generator=ge)
    W = DeviceWeights(header=h, rank=rank, n_ranks=n_ranks, n_heads=nh, n_kv_heads=nkv, ff_dim=ff0, vocab=v0, embedding=emb,
                      final_norm=norm(dim), wcls=q40(v0, dim, dim ** -0.5),
                      rope=torch.from_numpy(np.asarray(H.build_rope_table(h, h.seq_len))).to(device))
    n_exp = max(h.n_experts, 1)
    first_exp, n_local = (rank * (h.n_experts // n_ranks), h.n_experts // n_ranks) if ep else (0, n_exp)
    W.first_expert, W.n_local_experts, W.moe_mode = first_exp, (n_local if h.n_experts > 0 else 0), ("ep" if ep else "tp")
    gn = torch.Generator(device=device)
    gn.manual_seed(seed + 1)   # replicated tensors (norms, router gates)
    for _ in range(h.n_layers):
        L = LayerWeights(qkv=q40(q0 + 2 * kv0, dim, dim ** -0.5), wo=q40(dim, q0, 0.5 * (h.n_heads * hd) ** -0.5),
                         w13=q40(2 * ff0, dim, dim ** -0.5, lead=n_local), w2=q40(dim, ff0, 0.5 * h.ff_dim ** -0.5, lead=n_local),
                         norm0=(1.0 + 0.1 * torch.randn(dim, device=device, generator=gn)), norm1=(1.0 + 0.1 * torch.randn(dim, device=device, generator=gn)))
        if h.qk_norm:
            L.q_norm = 1.0 + 0.1 * torch.randn(hd, device=device, generator=gn)
            L.k_norm = 1.0 + 0.1 * torch.randn(hd, device=device, generator=gn)
        if h.n_experts > 0:
            L.moe_gate = torch.randn(h.n_experts, dim, device=device, generator=gn) * dim ** -0.5
        W.layers.append(L)
    torch.cuda.synchronize(device)
    W.bytes_uploaded = 0
    return W
