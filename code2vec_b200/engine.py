"""ctypes binding of libc2v_b200.so (include/c2v_b200.h) and the storage that goes with it.

PyTorch is used for device/pinned memory, streams and (elsewhere) torch.distributed only; every
arithmetic step of the hot path runs inside the C-ABI library's CUDA kernels.  There is no CPU
fallback: if the library cannot be loaded this module raises.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import Dict, Optional, Tuple

import numpy as np

from . import build as _build

PARAM_NAMES = ("tok", "path", "tgt", "W", "a")

MATH_FP32 = 0
MATH_TF32 = 1
MATH_3XTF32 = 2
MATH_MODES = {"fp32": MATH_FP32, "tf32": MATH_TF32, "3xtf32": MATH_3XTF32}


class c2v_dims(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("token_vocab", "path_vocab", "target_vocab", "embed_dim",
                                         "code_dim", "max_contexts", "max_batch", "top_k")]


class c2v_tensors(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in PARAM_NAMES]


class c2v_table_shards(C.Structure):
    _fields_ = [("world", C.c_int32), ("rank", C.c_int32), ("tok", C.c_void_p * 8), ("path", C.c_void_p * 8)]


class _DeviceArray:
    """A raw device allocation presented through __cuda_array_interface__ so torch can view it."""

    def __init__(self, ptr: int, shape):
        self.__cuda_array_interface__ = {"shape": tuple(int(x) for x in shape), "typestr": "<f4", "data": (int(ptr), False),
                                         "version": 2, "strides": None}


# every symbol include/c2v_b200.h declares: (restype, argtypes)
_P = C.c_void_p
_I32 = C.c_int32
_SIGNATURES = {
    "c2v_abi_version": (C.c_int, []),
    "c2v_last_error": (C.c_char_p, [_P]),
    "c2v_workspace_bytes": (C.c_size_t, [C.POINTER(c2v_dims)]),
    "c2v_create": (C.c_int, [C.POINTER(c2v_dims), C.c_int, C.POINTER(_P)]),
    "c2v_destroy": (None, [_P]),
    "c2v_bind_workspace": (C.c_int, [_P, _P, C.c_size_t]),
    "c2v_bind_params": (C.c_int, [_P, C.POINTER(c2v_tensors)]),
    "c2v_bind_grads": (C.c_int, [_P, C.POINTER(c2v_tensors)]),
    "c2v_bind_adam_state": (C.c_int, [_P, C.POINTER(c2v_tensors), C.POINTER(c2v_tensors)]),
    "c2v_set_option": (C.c_int, [_P, C.c_char_p, C.c_int64]),
    "c2v_get_option": (C.c_int, [_P, C.c_char_p, C.POINTER(C.c_int64)]),
    "c2v_forward": (C.c_int, [_P, _P, _P, _P, _P, _I32, _P, _P, _P]),
    "c2v_topk": (C.c_int, [_P, _P, _I32, _P, _P, _I32, _P]),
    "c2v_loss": (C.c_int, [_P, _P, _P, _I32, _P, _P]),
    "c2v_nearest_scratch_bytes": (C.c_size_t, [C.c_int64, _I32, _I32]),
    "c2v_compose_queries": (C.c_int, [_P, _P, C.c_int64, _I32, _P, _P, _P, _I32, _I32, _P, _P]),
    "c2v_nearest": (C.c_int, [_P, _P, C.c_int64, _I32, _P, _I32, _I32, _P, _I32, _P, _P, _P, C.c_size_t, _P]),
    "c2v_train_step": (C.c_int, [_P, _P, _P, _P, _P, _P, _I32, C.c_float, C.c_uint64, C.c_uint64, _P, _P, _P]),
    "c2v_sampled_train_step": (C.c_int, [_P, _P, _P, _P, _P, _P, _I32, _P, _I32, _P, _P, C.c_float,
                                         C.c_uint64, C.c_uint64, _P, _P, _P]),
    "c2v_adam_step": (C.c_int, [_P, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int64, _P]),
    "c2v_arm_target_adam": (C.c_int, [_P, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int64]),
    "c2v_hint_next_batch": (C.c_int, [_P, _P, _P, _P, _I32]),
    "c2v_hint_next_batch_host": (C.c_int, [_P, _P, _P, _P, _I32, _P]),
    "c2v_adam_step_range": (C.c_int, [_P, _P, _P, _P, _P, C.c_size_t, C.c_float, C.c_float, C.c_float, C.c_float,
                                      C.c_int64, _I32, _P]),
    "c2v_bind_table_shards": (C.c_int, [_P, C.POINTER(c2v_table_shards), C.POINTER(c2v_table_shards), C.c_float]),
    "c2v_scatter_inbox_bytes": (C.c_size_t, [C.POINTER(c2v_dims), _I32]),
    "c2v_bind_scatter_inbox": (C.c_int, [_P, C.POINTER(_P), _I32, _I32]),
    "c2v_apply_scatter_inbox": (C.c_int, [_P, _P]),
    "c2v_ipc_alloc": (C.c_int, [C.c_int, C.c_size_t, C.POINTER(_P), C.c_char_p]),
    "c2v_ipc_open": (C.c_int, [C.c_int, C.c_char_p, C.POINTER(_P)]),
    "c2v_ipc_close": (C.c_int, [C.c_int, _P]),
    "c2v_ipc_free": (C.c_int, [C.c_int, _P]),
    "c2v_train_batch_host": (C.c_int, [_P, _P, _P, _P, _P, _P, _I32, C.c_float, C.c_uint64, C.c_int64,
                                       C.c_float, C.c_float, C.c_float, C.c_float, _P, _P]),
    "c2v_train_batch_async": (C.c_int, [_P, _P, _P, _P, _P, _P, _I32, C.c_float, C.c_uint64, C.c_int64,
                                        C.c_float, C.c_float, C.c_float, C.c_float, _P, _P, _P]),
    "c2v_predict_batch_host": (C.c_int, [_P, _P, _P, _P, _P, _I32, _I32, _P, _P, _P, _P, _P]),
    "c2v_selftest_gemm": (C.c_int, [_P, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _P, C.c_size_t, _P, C.c_size_t,
                                    _P, C.c_size_t, _P]),
    "c2v_selftest_gemm3": (C.c_int, [_P, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _P, _P, C.c_size_t, _P, _P, C.c_size_t,
                                     _P, C.c_size_t, _P]),
    "c2v_selftest_split": (C.c_int, [_P, _P, _P, _P, C.c_size_t, _P]),
    "c2v_set_event": (C.c_int, [_P, C.c_char_p, _P]),
    "c2v_sync_tables": (C.c_int, [_P, _P]),
    "c2v_context_forward": (C.c_int, [_P, _P, _P, _P, _P, _I32, C.c_float, C.c_uint64, C.c_uint64, _P, _P, _P]),
    "c2v_target_forward": (C.c_int, [_P, _P, _I32, _P, _I32, _P, _P, _P, _P]),
    "c2v_lse_combine": (C.c_int, [_P, _P, _P, _I32, _I32, _P, C.c_float, _P, _P, _P]),
    "c2v_target_backward": (C.c_int, [_P, _P, _I32, _P, _P, _I32, C.c_float, _P, _P]),
    "c2v_context_backward": (C.c_int, [_P, _P, _P, _P, _P, _I32, C.c_float, C.c_uint64, C.c_uint64, _P, _P, _P]),
    "c2v_launch_count": (C.c_int64, [_P]),
    "c2v_phase_count": (C.c_int, []),
    "c2v_phase_name": (C.c_char_p, [C.c_int]),
    "c2v_phase_stats": (C.c_int, [_P, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.c_int]),
}

_lib = None


def library_path() -> str:
    return _build.LIB_PATH


def load_library():
    """Loads (building first if the in-tree .so is missing or stale) and types the C ABI."""
    global _lib
    if _lib is not None:
        return _lib
    if _build.needs_build():
        _build.build()
    if not os.path.exists(_build.LIB_PATH):
        raise RuntimeError("libc2v_b200.so is missing; run `python -m code2vec_b200.build`")
    lib = C.CDLL(_build.LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the header and the library disagree
        fn.restype = res
        fn.argtypes = args
    if lib.c2v_abi_version() != 1:
        raise RuntimeError("libc2v_b200.so ABI version mismatch")
    _lib = lib
    return lib


class EngineError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("c2v error %d: %s" % (code, msg))
        self.code = code


@dataclass
class EngineDims:
    token_vocab: int
    path_vocab: int
    target_vocab: int
    embed_dim: int
    code_dim: int
    max_contexts: int
    max_batch: int
    top_k: int = 10

    def shapes(self) -> Dict[str, Tuple[int, ...]]:
        d, D = self.embed_dim, self.code_dim
        return {"tok": (self.token_vocab, d), "path": (self.path_vocab, d), "tgt": (self.target_vocab, D),
                "W": (3 * d, D), "a": (D,)}

    def to_c(self) -> c2v_dims:
        return c2v_dims(self.token_vocab, self.path_vocab, self.target_vocab, self.embed_dim, self.code_dim,
                        self.max_contexts, self.max_batch, self.top_k)


def _ptr(t) -> Optional[int]:
    return None if t is None else t.data_ptr()


class PathAttentionEngine:
    """Owns the storage (torch tensors) and one c2v_engine handle on one GPU."""

    def __init__(self, dims: EngineDims, device: int = 0, training: bool = True):
        import torch
        if not torch.cuda.is_available():
            raise RuntimeError("PathAttentionEngine needs a CUDA device (B200); no CPU fallback exists")
        self.torch = torch
        self.lib = load_library()
        self.dims = dims
        self.device = int(device)
        self.dev = torch.device("cuda", self.device)
        self.training = training
        cd = dims.to_c()
        h = _P()
        rc = self.lib.c2v_create(C.byref(cd), self.device, C.byref(h))
        if rc != 0:
            raise EngineError(rc, self.lib.c2v_last_error(None).decode())
        self.h = h
        f32 = torch.float32
        with torch.cuda.device(self.dev):
            wbytes = self.lib.c2v_workspace_bytes(C.byref(cd))
            self.workspace = torch.empty(wbytes, dtype=torch.uint8, device=self.dev)
            self._check(self.lib.c2v_bind_workspace(self.h, self.workspace.data_ptr(), wbytes))
            # One flat fp32 buffer per role (parameters, gradients, Adam m, Adam v) with the five
            # tensors as views at 256-byte-aligned offsets: a data-parallel run can then
            # reduce-scatter / all-gather the whole model in one collective and run Adam on a slice.
            self.flat_params, self.params = self._alloc_flat()
            self._check(self.lib.c2v_bind_params(self.h, C.byref(self._tensors(self.params))))
            self.grads = self.adam_m = self.adam_v = None
            self.flat_grads = self.flat_m = self.flat_v = None
            if training:
                self.flat_grads, self.grads = self._alloc_flat()
                self.flat_m, self.adam_m = self._alloc_flat()
                self.flat_v, self.adam_v = self._alloc_flat()
                self._check(self.lib.c2v_bind_grads(self.h, C.byref(self._tensors(self.grads))))
                self._check(self.lib.c2v_bind_adam_state(self.h, C.byref(self._tensors(self.adam_m)),
                                                         C.byref(self._tensors(self.adam_v))))
            self._loss = torch.zeros(1, dtype=f32, device=self.dev)
        self.adam_t = 0

    # ---- plumbing -------------------------------------------------------------------------
    FLAT_ALIGN = 1024          # floats: keeps every view 256-byte aligned and any world size <= 256 dividing the total

    FLAT_ORDER = ("tgt", "tok", "path", "W", "a")   # target table first: its gradient is complete first (bucket A)

    def flat_layout(self):
        """[(name, offset, numel)] of the five tensors inside a flat buffer, and its padded length."""
        out, off = [], 0
        shapes = self.dims.shapes()
        for k in self.FLAT_ORDER:
            n = int(np.prod(shapes[k]))
            out.append((k, off, n))
            off = (off + n + self.FLAT_ALIGN - 1) // self.FLAT_ALIGN * self.FLAT_ALIGN
        return out, off

    def bucket_bounds(self):
        """Two gradient buckets of the flat buffer: A = target table (ready right after the dY GEMM),
        B = token/path tables, TRANSFORM, ATTENTION (ready at the end of the backward pass)."""
        layout, total = self.flat_layout()
        split = layout[1][1]            # offset of the first tensor after `tgt`
        return (0, split), (split, total)

    def set_event(self, name: str, event) -> None:
        """Ask the engine to record `event` (torch.cuda.Event) on the launching stream at a named point
        of c2v_train_step ("target_grads_ready": right after dY is complete)."""
        event.record(self.torch.cuda.current_stream(self.dev))          # forces creation of the cudaEvent_t
        self._events = getattr(self, "_events", {})
        self._events[name] = event
        self._check(self.lib.c2v_set_event(self.h, name.encode(), event.cuda_event))

    def _alloc_flat(self):
        torch = self.torch
        layout, total = self.flat_layout()
        flat = torch.zeros(total, dtype=torch.float32, device=self.dev)
        shp = self.dims.shapes()
        views = {k: flat[off:off + n].view(shp[k]) for k, off, n in layout}
        return flat, views

    @staticmethod
    def _tensors(d) -> c2v_tensors:
        return c2v_tensors(*[d[k].data_ptr() for k in PARAM_NAMES])

    def _check(self, rc: int):
        if rc != 0:
            raise EngineError(rc, self.lib.c2v_last_error(self.h).decode())

    def _stream(self) -> int:
        return self.torch.cuda.current_stream(self.dev).cuda_stream

    def close(self):
        if getattr(self, "h", None):
            self.lib.c2v_destroy(self.h)
            self.h = None
            # peers' shards first (unmap), then this rank's own allocations
            for p in getattr(self, "_ipc_opened", []):
                self.lib.c2v_ipc_close(self.device, p)
            self._ipc_opened = []
            self.shard_params = self.shard_grads = None          # views of the allocations freed below
            for p in getattr(self, "_ipc_owned", []):
                self.lib.c2v_ipc_free(self.device, p)
            self._ipc_owned = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, key: str, value: int):
        self._check(self.lib.c2v_set_option(self.h, key.encode(), int(value)))

    def get_option(self, key: str) -> int:
        v = C.c_int64()
        self._check(self.lib.c2v_get_option(self.h, key.encode(), C.byref(v)))
        return v.value

    @property
    def launch_count(self) -> int:
        return int(self.lib.c2v_launch_count(self.h))

    def selftest_split(self, x):
        """Test hook: the 3xTF32 operand split of a device tensor -> (hi, lo)."""
        hi, lo = self.torch.empty_like(x), self.torch.empty_like(x)
        self._check(self.lib.c2v_selftest_split(self.h, x.data_ptr(), hi.data_ptr(), lo.data_ptr(), x.numel(), self._stream()))
        return hi, lo

    def selftest_gemm(self, A, B, a_mn: bool, b_mn: bool, M: int, N: int, K: int, bn: int = 192, splits: int = 1,
                      three: bool = False):
        """Test hook: C[M,N] = A.B on the tcgen05 path.  A is [M,K] (a_mn False) or [K,M] (True) row-major,
        B is [N,K] (b_mn False) or [K,N] (True); returns C (slices summed on the host side of the test).
        three: as 3xTF32 (operands split on the device first)."""
        torch = self.torch
        out = torch.zeros((max(splits, 1), M, N), dtype=torch.float32, device=self.dev)
        if three:
            (Ah, Al), (Bh, Bl) = self.selftest_split(A), self.selftest_split(B)
            rc = self.lib.c2v_selftest_gemm3(self.h, int(a_mn), int(b_mn), bn, M, N, K, splits, Ah.data_ptr(), Al.data_ptr(),
                                             A.stride(0), Bh.data_ptr(), Bl.data_ptr(), B.stride(0), out.data_ptr(), N,
                                             self._stream())
        else:
            rc = self.lib.c2v_selftest_gemm(self.h, int(a_mn), int(b_mn), bn, M, N, K, splits, A.data_ptr(), A.stride(0),
                                            B.data_ptr(), B.stride(0), out.data_ptr(), N, self._stream())
        if rc < 0:
            self._check(rc)
        return out[:rc].sum(dim=0)

    def phase_stats(self, reset: bool = False) -> Dict[str, Tuple[float, int]]:
        """{phase name: (total device ms, number of timed occurrences)} since the last reset
        (needs set_option("profile", 1)).  Synchronises the device."""
        out = {}
        for i in range(self.lib.c2v_phase_count()):
            ms, n = C.c_double(), C.c_int64()
            self._check(self.lib.c2v_phase_stats(self.h, i, C.byref(ms), C.byref(n), 1 if reset else 0))
            if n.value:
                out[self.lib.c2v_phase_name(i).decode()] = (ms.value, n.value)
        return out

    # ---- parameters -----------------------------------------------------------------------
    def init_params(self, seed: int = 4321, scheme: str = "tensorflow"):
        """The reference's initialisers.  scheme "tensorflow" (tensorflow_model.py:205-220,249-250): tables
        U(+-sqrt(3/cols)) (variance_scaling fan_out uniform), TRANSFORM / ATTENTION glorot-uniform.
        scheme "keras" (keras_model.py:46-70, keras_attention_layer.py:29-34): embeddings and the attention
        vector U(+-0.05), both Dense kernels glorot-uniform (the output kernel is [D, |Y|] there).
        Drawn on the device with torch's generator (initialisation is not the hot path)."""
        torch = self.torch
        g = torch.Generator(device=self.dev)
        g.manual_seed(seed)
        d, D, Y = self.dims.embed_dim, self.dims.code_dim, self.dims.target_vocab
        if scheme == "tensorflow":
            lim = {"tok": (3.0 / d) ** 0.5, "path": (3.0 / d) ** 0.5, "tgt": (3.0 / D) ** 0.5,
                   "W": (6.0 / (3 * d + D)) ** 0.5, "a": (6.0 / (D + 1)) ** 0.5}
        elif scheme == "keras":
            lim = {"tok": 0.05, "path": 0.05, "tgt": (6.0 / (D + Y)) ** 0.5, "W": (6.0 / (3 * d + D)) ** 0.5, "a": 0.05}
        else:
            raise ValueError("unknown initialisation scheme: %r" % (scheme,))
        for k in PARAM_NAMES:
            self.params[k].uniform_(-lim[k], lim[k], generator=g)

    def load_params(self, arrays: Dict[str, np.ndarray]):
        torch = self.torch
        for k in PARAM_NAMES:
            src = torch.from_numpy(np.ascontiguousarray(arrays[k], dtype=np.float32))
            if tuple(src.shape) != tuple(self.params[k].shape):
                raise ValueError("parameter %s has shape %s, expected %s" % (k, tuple(src.shape), tuple(self.params[k].shape)))
            self.params[k].copy_(src)

    def sync_tables(self):
        """Lazy Adam: replay deferred updates so the parameter tensors can be read from outside the engine."""
        self._check(self.lib.c2v_sync_tables(self.h, self._stream()))

    def export_params(self) -> Dict[str, np.ndarray]:
        if getattr(self, "table_world", 1) > 1:
            # the token / path tables live in row shards (export_table_shards: this rank's rows); the replicated
            # tensors of the same name are stale and are not handed out
            return {k: self.params[k].detach().cpu().numpy() for k in ("tgt", "W", "a")}
        self.sync_tables()
        return {k: self.params[k].detach().cpu().numpy() for k in PARAM_NAMES}

    def export_grads(self) -> Dict[str, np.ndarray]:
        return {k: self.grads[k].detach().cpu().numpy() for k in PARAM_NAMES}

    def reset_optimizer(self):
        self.sync_tables()
        for d in (self.adam_m, self.adam_v):
            for t in d.values():
                t.zero_()
        self.adam_t = 0
        self.set_option("adam_step_count", 0)

    def to_device(self, arr, dtype):
        torch = self.torch
        if isinstance(arr, torch.Tensor):
            return arr.to(device=self.dev, dtype=dtype).contiguous()
        return torch.from_numpy(np.ascontiguousarray(arr)).to(device=self.dev, dtype=dtype)

    # ---- device-pointer entry points ---------------------------------------------------------
    def forward(self, src, path, tgt, mask, want_attention: bool = True):
        """c2v_forward: (code_vectors [B, D], attention [B, C] or None) as device tensors."""
        torch = self.torch
        B, Cn = src.shape
        code = torch.empty((B, self.dims.code_dim), dtype=torch.float32, device=self.dev)
        attn = torch.empty((B, Cn), dtype=torch.float32, device=self.dev) if want_attention else None
        self._check(self.lib.c2v_forward(self.h, src.data_ptr(), path.data_ptr(), tgt.data_ptr(), mask.data_ptr(),
                                         B, code.data_ptr(), _ptr(attn), self._stream()))
        return code, attn

    def topk(self, code_vec, normalize: bool = False):
        torch = self.torch
        B = code_vec.shape[0]
        k = min(self.dims.top_k, self.dims.target_vocab)
        idx = torch.empty((B, k), dtype=torch.int32, device=self.dev)
        val = torch.empty((B, k), dtype=torch.float32, device=self.dev)
        self._check(self.lib.c2v_topk(self.h, code_vec.data_ptr(), B, idx.data_ptr(), val.data_ptr(),
                                      int(normalize), self._stream()))
        return idx, val

    # ---- nearest-neighbour search (c2v_compose_queries / c2v_nearest) ---------------------------------
    NEAREST_MAX_K = 64
    NEAREST_MAX_EXCLUDE = 16
    MAX_QUERY_TERMS = 16

    @staticmethod
    def nearest_query_capacity(dim: int) -> int:
        """Queries c2v_nearest keeps in shared memory per chunk at this width (similarity.cuh, query_capacity): the
        bank is read once per chunk."""
        return min(64, max(8, (32768 // (int(dim) * 4)) // 8 * 8))

    def compose_queries(self, bank, terms):
        """gensim's query vectors for word queries: terms = one list per query of (row or vector, weight) pairs, a row
        being an int index into `bank` (unit-normalised before weighting) and a vector a 1-D array / tensor of
        bank.shape[1] floats used as given.  Returns a device tensor [n, dim] of unit vectors (c2v_compose_queries)."""
        torch = self.torch
        n, dim = len(terms), int(bank.shape[1])
        mt = max([len(t) for t in terms] + [1])
        if mt > self.MAX_QUERY_TERMS:
            raise ValueError("at most %d terms per query" % self.MAX_QUERY_TERMS)
        rows = np.full((n, mt), -1, dtype=np.int32)
        weights = np.zeros((n, mt), dtype=np.float32)
        vecs = None
        for q, query in enumerate(terms):
            for t, (term, w) in enumerate(query):
                weights[q, t] = float(w)
                if isinstance(term, (int, np.integer)):
                    if not 0 <= int(term) < bank.shape[0]:
                        raise IndexError("row %d outside the bank (%d rows)" % (int(term), bank.shape[0]))
                    rows[q, t] = int(term)
                else:
                    v = np.asarray(term.detach().cpu() if hasattr(term, "detach") else term, dtype=np.float32).reshape(-1)
                    if v.shape[0] != dim:
                        raise ValueError("query vector has %d elements, the bank has %d columns" % (v.shape[0], dim))
                    if vecs is None:
                        vecs = np.zeros((n, mt, dim), dtype=np.float32)
                    vecs[q, t] = v
                    rows[q, t] = -2
        out = torch.empty((n, dim), dtype=torch.float32, device=self.dev)
        d_rows, d_w = self.to_device(rows, torch.int32), self.to_device(weights, torch.float32)
        d_vecs = None if vecs is None else self.to_device(vecs, torch.float32)
        self._check(self.lib.c2v_compose_queries(self.h, bank.data_ptr(), int(bank.shape[0]), dim, d_rows.data_ptr(),
                                                 d_w.data_ptr(), _ptr(d_vecs), n, mt, out.data_ptr(), self._stream()))
        return out

    def nearest(self, bank, queries, k: int, exclude=None):
        """Cosine top-k of the rows of `bank` (device [rows, dim] float32) for each query (device [n, dim]):
        (idx int32 [n, k], val float32 [n, k]) device tensors, score descending, ties to the lower row; slots beyond
        the available results hold -1 / -inf.  exclude: [n, <= 16] row ids never returned (-1 = padding)."""
        torch = self.torch
        bank = bank if bank.is_contiguous() else bank.contiguous()
        queries = self.to_device(queries, torch.float32)
        if queries.dim() == 1:
            queries = queries.view(1, -1)
        n, dim = int(queries.shape[0]), int(bank.shape[1])
        ex, n_ex = None, 0
        if exclude is not None:
            ex = self.to_device(exclude, torch.int32)
            if ex.dim() != 2 or ex.shape[0] != n:
                raise ValueError("exclude must be [n, n_exclude]")
            n_ex = int(ex.shape[1])
            if n_ex == 0:
                ex = None
        idx = torch.empty((n, k), dtype=torch.int32, device=self.dev)
        val = torch.empty((n, k), dtype=torch.float32, device=self.dev)
        nbytes = int(self.lib.c2v_nearest_scratch_bytes(int(bank.shape[0]), n, int(k)))
        scratch = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=self.dev)
        self._check(self.lib.c2v_nearest(self.h, bank.data_ptr(), int(bank.shape[0]), dim, queries.data_ptr(), n, int(k),
                                         _ptr(ex), n_ex, idx.data_ptr(), val.data_ptr(), scratch.data_ptr(), nbytes,
                                         self._stream()))
        return idx, val

    def loss(self, code_vec, target):
        out = self.torch.empty(1, dtype=self.torch.float32, device=self.dev)
        self._check(self.lib.c2v_loss(self.h, code_vec.data_ptr(), target.data_ptr(), code_vec.shape[0],
                                      out.data_ptr(), self._stream()))
        return out

    def train_step(self, src, path, tgt, mask, target, keep: float = 1.0, seed: int = 0, step: int = 0,
                   dropout_mask=None, loss_out=None):
        out = self._loss if loss_out is None else loss_out
        self._check(self.lib.c2v_train_step(self.h, src.data_ptr(), path.data_ptr(), tgt.data_ptr(), mask.data_ptr(),
                                            target.data_ptr(), src.shape[0], float(keep), int(seed), int(step),
                                            _ptr(dropout_mask), out.data_ptr(), self._stream()))
        return out

    def sampled_train_step(self, src, path, tgt, mask, target, sampled, logq_true, logq_sampled, keep: float = 1.0,
                           seed: int = 0, step: int = 0, dropout_mask=None, loss_out=None):
        out = self._loss if loss_out is None else loss_out
        self._check(self.lib.c2v_sampled_train_step(
            self.h, src.data_ptr(), path.data_ptr(), tgt.data_ptr(), mask.data_ptr(), target.data_ptr(),
            src.shape[0], sampled.data_ptr(), sampled.shape[0], logq_true.data_ptr(), logq_sampled.data_ptr(),
            float(keep), int(seed), int(step), _ptr(dropout_mask), out.data_ptr(), self._stream()))
        return out

    def adam_step(self, lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-8, t: Optional[int] = None):
        if t is None:
            self.adam_t += 1
            t = self.adam_t
        else:
            self.adam_t = t
        self._check(self.lib.c2v_adam_step(self.h, lr, beta1, beta2, eps, int(t), self._stream()))

    def arm_target_adam(self, t: int, lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-8):
        """The next train step's dY epilogue applies Adam step `t` to the target table (c2v_arm_target_adam);
        the following adam_step(t) skips that table.  The target gradient buffer is then not written."""
        self._check(self.lib.c2v_arm_target_adam(self.h, lr, beta1, beta2, eps, int(t)))

    def hint_next_batch(self, src, path, tgt):
        """Device index tensors [B, C] of the batch the next train step will use (c2v_hint_next_batch); the
        caller keeps them alive until that step has been issued."""
        self._check(self.lib.c2v_hint_next_batch(self.h, src.data_ptr(), path.data_ptr(), tgt.data_ptr(), int(src.shape[0])))

    def hint_next_batch_host(self, src, path, tgt):
        """Same from host arrays / pinned tensors (c2v_hint_next_batch_host)."""
        src, path, tgt = (_as_host(x, np.int32) for x in (src, path, tgt))      # pageable sources are staged before the call returns
        self._check(self.lib.c2v_hint_next_batch_host(self.h, _host_ptr(src), _host_ptr(path), _host_ptr(tgt),
                                                      int(src.shape[0]), self._stream()))

    def adam_step_range(self, theta, grad, m, v, t: int, lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-8, zero_grad=False):
        """TF1 Adam on one contiguous slice (the sharded-optimizer path): flat tensors of equal length."""
        n = int(theta.numel())
        assert grad.numel() == n and m.numel() == n and v.numel() == n
        self.adam_t = int(t)
        self._check(self.lib.c2v_adam_step_range(self.h, theta.data_ptr(), grad.data_ptr(), m.data_ptr(), v.data_ptr(),
                                                 n, lr, beta1, beta2, eps, int(t), 1 if zero_grad else 0, self._stream()))

    # ---- phase-split step (fully sharded schedule) ------------------------------------------------
    def context_forward(self, src, path, tgt, mask, code_out, keep=1.0, seed=0, step=0, dropout_mask=None):
        self._check(self.lib.c2v_context_forward(self.h, src.data_ptr(), path.data_ptr(), tgt.data_ptr(), mask.data_ptr(),
                                                 src.shape[0], float(keep), int(seed), int(step), _ptr(dropout_mask),
                                                 code_out.data_ptr(), self._stream()))

    def target_forward(self, code_all, target_all, row_offset, row_max, row_sum, true_logit):
        self._check(self.lib.c2v_target_forward(self.h, code_all.data_ptr(), code_all.shape[0], target_all.data_ptr(),
                                                int(row_offset), row_max.data_ptr(), row_sum.data_ptr(),
                                                true_logit.data_ptr(), self._stream()))

    def lse_combine(self, maxes, sums, true_logit, lse_out, loss_out):
        world, Bt = maxes.shape
        self._check(self.lib.c2v_lse_combine(self.h, maxes.data_ptr(), sums.data_ptr(), world, Bt, true_logit.data_ptr(),
                                             1.0 / Bt, lse_out.data_ptr(), loss_out.data_ptr(), self._stream()))

    def target_backward(self, code_all, lse, target_all, row_offset, dv_partial):
        Bt = code_all.shape[0]
        self._check(self.lib.c2v_target_backward(self.h, code_all.data_ptr(), Bt, lse.data_ptr(), target_all.data_ptr(),
                                                 int(row_offset), 1.0 / Bt, dv_partial.data_ptr(), self._stream()))

    def context_backward(self, src, path, tgt, mask, dv, keep=1.0, seed=0, step=0, dropout_mask=None):
        self._check(self.lib.c2v_context_backward(self.h, src.data_ptr(), path.data_ptr(), tgt.data_ptr(), mask.data_ptr(),
                                                  src.shape[0], float(keep), int(seed), int(step), _ptr(dropout_mask),
                                                  dv.data_ptr(), self._stream()))

    # ---- row-sharded embedding tables over peer memory (data-parallel runs) ----------------------
    def apply_scatter_inbox(self):
        """Owner side of the push-based gradient exchange: fold this rank's inbox into its gradient shards (call after
        the cross-rank barrier that follows every rank's backward pass)."""
        self._check(self.lib.c2v_apply_scatter_inbox(self.h, self._stream()))

    def enable_table_sharding(self, group=None, push_grads: bool = False):
        """Re-homes WORDS_VOCAB / PATHS_VOCAB (+ gradients, Adam slots) as row-interleaved shards: global
        row r -> rank r % world, local row r // world.  Parameter and gradient shards live in
        cudaMalloc'ed memory whose CUDA-IPC handles are exchanged once, so every rank's kernels can
        load rows from, and red.add gradients into, every other rank's shard over NVLink.  The current
        contents of the replicated tables are carried over."""
        import torch.distributed as dist
        torch = self.torch
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        if world not in (1, 2, 4, 8):
            raise ValueError("table sharding needs a world size of 1, 2, 4 or 8")
        if self.training and self.get_option("lazy_adam"):
            self.set_option("lazy_adam", 0)          # flushes deferred updates; shards use the dense per-rank Adam
        d = self.dims.embed_dim
        rows = {"tok": (self.dims.token_vocab + world - 1) // world, "path": (self.dims.path_vocab + world - 1) // world}
        own, handles = {}, {}
        self.push_grads = bool(push_grads) and self.training and world > 1
        if self.push_grads:          # one inbox per rank for the embedding-gradient rows its peers push (c2v_bind_scatter_inbox)
            cd = self.dims.to_c()
            nbytes = self.lib.c2v_scatter_inbox_bytes(C.byref(cd), world)
            ptr, hbuf = _P(), C.create_string_buffer(64)
            rc = self.lib.c2v_ipc_alloc(self.device, nbytes, C.byref(ptr), hbuf)
            if rc != 0:
                raise EngineError(rc, self.lib.c2v_last_error(None).decode())
            own[("inbox", "all")] = ptr.value
            handles[("inbox", "all")] = hbuf.raw
        for role in ("params", "grads"):
            for name in ("tok", "path"):
                ptr, hbuf = _P(), C.create_string_buffer(64)
                rc = self.lib.c2v_ipc_alloc(self.device, rows[name] * d * 4, C.byref(ptr), hbuf)
                if rc != 0:
                    raise EngineError(rc, self.lib.c2v_last_error(None).decode())
                own[(role, name)] = ptr.value
                handles[(role, name)] = hbuf.raw
        gathered = [None] * world
        dist.all_gather_object(gathered, handles, group=group)
        ptrs = {}
        self._ipc_opened = []
        for r in range(world):
            for key in handles:
                if r == rank:
                    ptrs[(r,) + key] = own[key]
                else:
                    p = _P()
                    rc = self.lib.c2v_ipc_open(self.device, gathered[r][key], C.byref(p))
                    if rc != 0:
                        raise EngineError(rc, self.lib.c2v_last_error(None).decode())
                    ptrs[(r,) + key] = p.value
                    self._ipc_opened.append(p.value)
        self._ipc_owned = list(own.values())

        def shards(role):
            st = c2v_table_shards()
            st.world, st.rank = world, rank
            for r in range(world):
                st.tok[r] = ptrs[(r, role, "tok")]
                st.path[r] = ptrs[(r, role, "path")]
            return st

        sp, sg = shards("params"), shards("grads")
        self._check(self.lib.c2v_bind_table_shards(self.h, C.byref(sp), C.byref(sg) if self.training else None, 1.0 / world))
        if self.push_grads:
            arr = (_P * world)(*[ptrs[(r, "inbox", "all")] for r in range(world)])
            self._check(self.lib.c2v_bind_scatter_inbox(self.h, arr, world, rank))
        view = lambda key, name: torch.as_tensor(_DeviceArray(own[key], (rows[name], d)), device=self.dev)
        self.table_world, self.table_rank = world, rank
        self.shard_params = {n: view(("params", n), n) for n in ("tok", "path")}
        self.shard_grads = {n: view(("grads", n), n) for n in ("tok", "path")}
        self.shard_m = {n: torch.zeros((rows[n], d), dtype=torch.float32, device=self.dev) for n in ("tok", "path")}
        self.shard_v = {n: torch.zeros((rows[n], d), dtype=torch.float32, device=self.dev) for n in ("tok", "path")}
        for n in ("tok", "path"):
            mine = self.params[n][rank::world]
            self.shard_params[n][:mine.shape[0]].copy_(mine)
        torch.cuda.synchronize(self.dev)
        dist.barrier(group=group)

    def load_table_shards(self, arrays: Dict[str, np.ndarray]):
        """Fill this rank's shards from full [T, d] / [P, d] host tables."""
        torch = self.torch
        for n in ("tok", "path"):
            mine = np.ascontiguousarray(arrays[n][self.table_rank::self.table_world], dtype=np.float32)
            self.shard_params[n][:mine.shape[0]].copy_(torch.from_numpy(mine))

    def export_table_shards(self) -> Dict[str, np.ndarray]:
        return {n: self.shard_params[n].detach().cpu().numpy() for n in ("tok", "path")}

    # ---- host-buffer entry points ------------------------------------------------------------
    def train_batch_host(self, src, path, tgt, mask, target, keep: float = 1.0, seed: int = 0,
                         lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-8) -> float:
        """One reference `sess.run([optimizer, train_loss])` on HOST arrays (numpy or pinned torch
        tensors): H2D copies, train step, Adam, loss read-back -- all inside the C-ABI call."""
        loss = np.zeros(1, dtype=np.float32)
        B = int(src.shape[0])
        src, path, tgt, target = (_as_host(x, np.int32) for x in (src, path, tgt, target))
        mask = _as_host(mask, np.float32)
        self._check(self.lib.c2v_train_batch_host(
            self.h, _host_ptr(src), _host_ptr(path), _host_ptr(tgt), _host_ptr(mask), _host_ptr(target), B,
            float(keep), int(seed), int(self.adam_t + 1), lr, beta1, beta2, eps, loss.ctypes.data, self._stream()))
        self.adam_t += 1          # only once the step went through: a failed call leaves host and engine counters in step
        return float(loss[0])

    def train_batch_async(self, src, path, tgt, mask, target, rows: int, loss_out, upload_done=None, keep: float = 1.0,
                          seed: int = 0, lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-8):
        """c2v_train_batch_async on PINNED torch tensors (first `rows` rows): the upload runs on the engine's copy stream,
        the step is queued behind it, nothing is waited for.  loss_out: pinned float32 tensor of one element; upload_done:
        torch.cuda.Event recorded when the inputs have left the host buffers."""
        for x in (src, path, tgt, mask, target, loss_out):
            if not x.is_pinned():
                raise ValueError("c2v_train_batch_async needs page-locked host tensors")
        ev = None
        if upload_done is not None:
            upload_done.record(self.torch.cuda.current_stream(self.dev))      # forces creation of the cudaEvent_t; re-recorded by the engine
            ev = upload_done.cuda_event
        self._check(self.lib.c2v_train_batch_async(
            self.h, src.data_ptr(), path.data_ptr(), tgt.data_ptr(), mask.data_ptr(), target.data_ptr(), int(rows),
            float(keep), int(seed), int(self.adam_t + 1), lr, beta1, beta2, eps, loss_out.data_ptr(), ev, self._stream()))
        self.adam_t += 1

    def predict_batch_host(self, src, path, tgt, mask, normalize: bool = False, want_code: bool = True,
                           want_attention: bool = True):
        B, Cn = int(src.shape[0]), int(src.shape[1])
        src, path, tgt = (_as_host(x, np.int32) for x in (src, path, tgt))
        mask = _as_host(mask, np.float32)
        k = min(self.dims.top_k, self.dims.target_vocab)
        idx = np.empty((B, k), dtype=np.int32)
        val = np.empty((B, k), dtype=np.float32)
        code = np.empty((B, self.dims.code_dim), dtype=np.float32) if want_code else None
        attn = np.empty((B, Cn), dtype=np.float32) if want_attention else None
        self._check(self.lib.c2v_predict_batch_host(
            self.h, _host_ptr(src), _host_ptr(path), _host_ptr(tgt), _host_ptr(mask), B, int(normalize),
            idx.ctypes.data, val.ctypes.data, None if code is None else code.ctypes.data,
            None if attn is None else attn.ctypes.data, self._stream()))
        return idx, val, code, attn


_TORCH_DTYPE_NAMES = {np.dtype(np.int32): "torch.int32", np.dtype(np.float32): "torch.float32"}


def _as_host(a, dtype):
    """numpy arrays are made contiguous/typed (no copy when already so); torch CPU tensors pass through, but only
    with the element type the C entry point reads -- an int64 index tensor read as int32 would index the tables
    out of range without any error."""
    if isinstance(a, np.ndarray):
        return np.ascontiguousarray(a, dtype=dtype)
    if hasattr(a, "dtype") and hasattr(a, "data_ptr"):
        want = _TORCH_DTYPE_NAMES[np.dtype(dtype)]
        if str(a.dtype) != want:
            raise TypeError("host tensor has dtype %s, the engine reads %s" % (a.dtype, want))
    return a


def _host_ptr(a) -> int:
    """Address of a contiguous host buffer: numpy array or (pinned) CPU torch tensor."""
    if isinstance(a, np.ndarray):
        if not a.flags["C_CONTIGUOUS"]:
            raise ValueError("host buffer must be C-contiguous")
        return a.ctypes.data
    if hasattr(a, "data_ptr"):
        if a.device.type != "cpu" or not a.is_contiguous():
            raise ValueError("host buffer must be a contiguous CPU tensor")
        return a.data_ptr()
    raise TypeError("unsupported host buffer type %r" % type(a))
