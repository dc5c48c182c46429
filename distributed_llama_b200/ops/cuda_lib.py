"""ctypes binding of the sm_100a kernel/runtime library (csrc/cuda -> distributed_llama_b200/_cuda.so).

The library is torch-free: tensors cross the boundary as raw device pointers + the current CUDA stream handle.
If the library is missing on a machine with a GPU we build it; failures are loud (no eager fallback).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

from .. import _build

_lib: Optional[C.CDLL] = None

u32, u64, i32, f32, vp = C.c_uint32, C.c_uint64, C.c_int, C.c_float, C.c_void_p


class EngineConfig(C.Structure):
    _fields_ = [(n, u32) for n in ("dim", "nLayers", "nHeads", "nKvHeads", "headDim", "ffDim", "vocab", "seqLen",
                                   "nExperts", "nActiveExperts", "maxBatch", "nSplits", "rank", "nRanks", "numSms")] + \
               [("eps", f32), ("usePdl", u32), ("moeFirstExpert", u32), ("moeNumLocal", u32), ("wType", u32), ("hiddenAct", u32),
                ("vocabFull", u32), ("maxPrefill", u32)]


class LayerPtrs(C.Structure):
    _fields_ = [(n, vp) for n in ("qkvQs", "qkvSc", "woQs", "woSc", "w13Qs", "w13Sc", "w2Qs", "w2Sc",
                                  "norm0", "norm1", "qNorm", "kNorm", "moeGate")]


class GlobalPtrs(C.Structure):
    _fields_ = [("embedding", vp), ("embeddingPeers", vp * 8), ("embRowsPerRank", u32), ("finalNorm", vp), ("wclsQs", vp), ("wclsSc", vp),
                ("rope", vp)]


class EngineBuffers(C.Structure):
    _fields_ = [(n, vp) for n in ("tokens", "pos", "history", "logits", "x", "pTokens", "pPos")] + \
               [("kCache", C.POINTER(vp)), ("vCache", C.POINTER(vp))] + \
               [(n, vp) for n in ("pTargets", "pLogprob", "pTopId", "pTopLogprob")]


class CommPtrs(C.Structure):
    _fields_ = [("arena", vp * 8), ("mcArena", vp)]


class _DeviceArray:
    def __init__(self, ptr: int, shape, typestr: str, owner):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (ptr, False), "version": 2}
        self.owner = owner


def device_view(ptr: int, shape, dtype, owner=None, device=None):
    """A torch tensor over device memory torch did not allocate. `owner` stays alive as long as the tensor or any view of it."""
    import torch
    typestr = {torch.float32: "<f4", torch.int32: "<i4", torch.bfloat16: "<i2"}[dtype]   # the interface has no bf16 type
    return torch.as_tensor(_DeviceArray(ptr, shape, typestr, owner), device=device).view(dtype)


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    path = _build.build_cuda()
    L = C.CDLL(str(path))
    L.dl_repack_q40.argtypes = [vp, u64, u64, u32, u32, vp, vp, u32, u32, u32, vp]
    L.dl_repack_q40.restype = i32
    L.dl_dequant_device_q40.argtypes = [vp, vp, u32, u32, vp, vp]
    L.dl_dequant_device_q40.restype = i32
    L.dl_gemv_q40.argtypes = [i32, i32, i32, vp, vp, u32, u32, vp, u32, vp, f32, vp, u32, i32, vp, i32, i32]
    L.dl_gemv_q40.restype = i32
    L.dl_gemv_dense.argtypes = [i32, i32, i32, i32, vp, u32, u32, vp, u32, vp, f32, vp, u32, i32, vp, i32]
    L.dl_gemv_dense.restype = i32
    L.dl_gemm_q40_tc.argtypes = [i32, vp, vp, u32, u32, vp, u32, u32, vp, u32, i32, vp, i32, i32]
    L.dl_gemm_q40_tc.restype = i32
    L.dl_rmsnorm_bf16.argtypes = [vp, u32, vp, vp, u32, u32, f32, u32, vp]
    L.dl_rmsnorm_bf16.restype = i32
    L.dl_attn_prefill_tc.argtypes = [vp, u32, u32, u32, u32, u32, u32, u32, vp, vp, vp, u32, vp]
    L.dl_attn_prefill_tc.restype = i32
    L.dl_engine_create.argtypes = [C.POINTER(EngineConfig)]
    L.dl_engine_create.restype = vp
    L.dl_engine_destroy.argtypes = [vp]
    L.dl_engine_destroy.restype = None
    L.dl_engine_set_layer.argtypes = [vp, u32, C.POINTER(LayerPtrs)]
    L.dl_engine_set_layer.restype = i32
    L.dl_engine_set_globals.argtypes = [vp, C.POINTER(GlobalPtrs)]
    L.dl_engine_set_globals.restype = i32
    L.dl_engine_get_config.argtypes = [vp, C.POINTER(EngineConfig)]
    L.dl_engine_get_config.restype = i32
    L.dl_engine_buffers.argtypes = [vp, C.POINTER(EngineBuffers)]
    L.dl_engine_buffers.restype = i32
    L.dl_engine_arena_bytes.argtypes = [C.POINTER(EngineConfig)]
    L.dl_engine_arena_bytes.restype = C.c_size_t
    L.dl_engine_enable_mega.argtypes = [vp, i32]
    L.dl_engine_enable_mega.restype = i32
    L.dl_engine_set_vocab_limit.argtypes = [vp, u32]
    L.dl_engine_set_vocab_limit.restype = i32
    L.dl_engine_set_comm.argtypes = [vp, C.POINTER(CommPtrs)]
    L.dl_engine_set_comm.restype = i32
    for name, args in (("dl_comm_alloc", [C.c_size_t, C.POINTER(vp)]), ("dl_comm_free", [vp]), ("dl_comm_ipc_handle", [vp, vp]),
                       ("dl_comm_ipc_open", [vp, C.POINTER(vp)]), ("dl_comm_ipc_close", [vp]), ("dl_comm_memset", [vp, i32, C.c_size_t, vp])):
        getattr(L, name).argtypes = args
        getattr(L, name).restype = i32
    L.dl_vmm_supported.argtypes = [C.POINTER(C.c_int)]
    L.dl_vmm_supported.restype = i32
    L.dl_vmm_create.argtypes = [u32, u32, C.c_size_t, C.c_char_p, i32]
    L.dl_vmm_create.restype = vp
    L.dl_vmm_connect.argtypes = [vp]
    L.dl_vmm_connect.restype = i32
    L.dl_vmm_ptr.argtypes = [vp, u32]
    L.dl_vmm_ptr.restype = vp
    L.dl_vmm_mc_ptr.argtypes = [vp]
    L.dl_vmm_mc_ptr.restype = vp
    L.dl_vmm_bytes.argtypes = [vp]
    L.dl_vmm_bytes.restype = C.c_size_t
    L.dl_vmm_destroy.argtypes = [vp]
    L.dl_vmm_destroy.restype = None
    L.dl_vmm_selftest_kernel.argtypes = [vp, u32, i32, vp]
    L.dl_vmm_selftest_kernel.restype = i32
    L.dl_engine_set_trace.argtypes = [vp, vp, u32]
    L.dl_engine_set_trace.restype = i32
    L.dl_engine_sampler_seed.argtypes = [vp, C.c_uint64]
    L.dl_engine_sampler_seed.restype = i32
    L.dl_engine_sample.argtypes = [vp, f32, f32, vp]
    L.dl_engine_sample.restype = i32
    L.dl_sample_logits.argtypes = [vp, vp, u32, f32, f32, vp, vp, vp]
    L.dl_sample_logits.restype = i32
    L.dl_engine_sync_ns.argtypes = [vp]
    L.dl_engine_sync_ns.restype = C.c_uint64
    L.dl_engine_mega_active.argtypes = [vp]
    L.dl_engine_mega_active.restype = i32
    L.dl_engine_aborted.argtypes = [vp]
    L.dl_engine_aborted.restype = i32
    L.dl_engine_set_trace_all.argtypes = [vp, i32]
    L.dl_engine_set_trace_all.restype = i32
    L.dl_engine_forward.argtypes = [vp, i32, i32, i32, vp]
    L.dl_engine_forward.restype = i32
    L.dl_engine_forward_part.argtypes = [vp, i32, u32, i32, vp, vp]
    L.dl_engine_forward_part.restype = i32
    L.dl_engine_prefill.argtypes = [vp, u32, u32, i32, vp]
    L.dl_engine_prefill.restype = i32
    L.dl_engine_score.argtypes = [vp, u32, u32, vp]
    L.dl_engine_score.restype = i32
    L.dl_engine_score_max_tokens.argtypes = [vp]
    L.dl_engine_score_max_tokens.restype = u32
    L.dl_score_rows.argtypes = [vp, u32, u32, u32, vp, u32, vp, vp, vp, vp]
    L.dl_score_rows.restype = i32
    L.dl_engine_capture_decode.argtypes = [vp]
    L.dl_engine_capture_decode.restype = i32
    L.dl_engine_decode_graph.argtypes = [vp, i32, vp]
    L.dl_engine_decode_graph.restype = i32
    _lib = L
    return L


_ERRORS = {
    -30: "tensor-parallel slice too narrow for the fused all-reduce GEMV: the per-rank K of WO / W2 (heads/N * headDim, ffDim/N) "
         "must be a multiple of 128 — use fewer ranks, or DL_COLLECTIVES=nccl",
    -31: "mixture-of-experts up-projection shape not covered by the TMA GEMV",
    -32: "mixture-of-experts down-projection shape not covered by the TMA GEMV (per-rank expert ffDim must be a multiple of 128: use moe_mode=ep)",
    -33: "arg-max under tensor parallelism needs the fused logits kernel",
    -36: "mixture-of-experts prefill shape not covered (dim, ffDim multiples of 256, chunk <= 256 tokens)",
    -37: "scoring under tensor parallelism needs the peer arena (fused collectives)",
}


def check(code: int, what: str) -> None:
    if code != 0:
        raise RuntimeError(f"{what} failed with code {code}" + (f": {_ERRORS[code]}" if code in _ERRORS else ""))


def stream_ptr() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream


PRO_RMSNORM, PRO_PLAIN = 0, 1
EPI_STORE, EPI_RESIDUAL, EPI_SWIGLU = 0, 1, 2
GEPI_STORE_F32, GEPI_RESIDUAL, GEPI_SWIGLU_BF16, GEPI_STORE_BF16 = 0, 1, 2, 3
