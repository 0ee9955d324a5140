"""ctypes binding of libvpca.so (include/vpca.h) -- the Python twin of the JNI class ``NativePca``
shown in INTEGRATION.md.  One ``NativePca`` object = one ``vpca_ctx`` = one GPU.

There is no CPU fallback: importing this module never fails (so host logic stays testable without a
GPU), but constructing ``NativePca`` raises ``VpcaError`` when the CUDA library is missing or no
sm_100 device is usable.
"""
from __future__ import annotations

import ctypes
import os
from pathlib import Path
from typing import Optional, Tuple

import numpy as np

VPCA_OK = 0
VPCA_ERR_BAD_ARG = -1
VPCA_ERR_INDEX_OUT_OF_RANGE = -2
VPCA_ERR_CUDA = -3
VPCA_ERR_NCCL = -4
VPCA_ERR_OVERFLOW = -5
VPCA_ERR_STATE = -6
VPCA_ERR_NOMEM = -7
VPCA_ERR_UNSUPPORTED = -8
JOIN, MERGE = 0, 1    # vpca_join_rows modes (VPCA_JOIN / VPCA_MERGE)

DTYPE_I8 = 0
DTYPE_BF16 = 1
DTYPE_E2M1 = 2   # 4-bit cells, two per byte (cell j of a row in nibble j & 1 of byte j // 2; value m is the code 2 m)

_STATUS_NAMES = {
    -1: "BAD_ARG", -2: "INDEX_OUT_OF_RANGE", -3: "CUDA", -4: "NCCL", -5: "OVERFLOW", -6: "STATE",
    -7: "NOMEM", -8: "UNSUPPORTED",
}

# every symbol include/vpca.h declares (checked by tests/test_abi.py against the header)
EXPORTED_SYMBOLS = (
    "vpca_version", "vpca_create", "vpca_destroy", "vpca_last_error", "vpca_reset", "vpca_encode_calls",
    "vpca_accumulate_calls", "vpca_commit", "vpca_abort", "vpca_accumulate_dense", "vpca_gram_device_ptr",
    "vpca_finalize_gram", "vpca_get_gram", "vpca_set_gram", "vpca_compute_pca", "vpca_get_centered",
    "vpca_get_tridiagonal", "vpca_synth_dense_device", "vpca_get_stats", "vpca_debug_gram_profile",
    "vpca_gram_export_ipc", "vpca_gram_set_peers", "vpca_peer_barrier", "vpca_accumulate_panels",
    "vpca_synth_panels_device", "vpca_accumulate_calls_u16", "vpca_get_partial_gram", "vpca_load_partial_gram",
    "vpca_accumulate_bits", "vpca_gram_set_peer_mode", "vpca_gram_gather", "vpca_accumulate_bed",
    "vpca_synchronize", "vpca_host_alloc", "vpca_host_free", "vpca_gram_set_peers_local", "vpca_owner_row_bands",
    "vpca_get_gram_band", "vpca_variant_count", "vpca_debug_rebalance",
    "vpca_debug_lanczos_profile", "vpca_debug_max_clusters", "vpca_debug_band_tiles", "vpca_hash_keys", "vpca_join_rows", "vpca_join_fetch", "vpca_join_size", "vpca_accumulate_joined",
    "vpca_pool_create", "vpca_pool_destroy", "vpca_pool_size", "vpca_pool_ctx", "vpca_pool_last_error", "vpca_pool_reset",
    "vpca_pool_accumulate_calls", "vpca_pool_accumulate_calls_u16", "vpca_pool_accumulate_bits", "vpca_pool_accumulate_bed",
    "vpca_pool_commit", "vpca_pool_abort", "vpca_pool_reduce_and_finalize", "vpca_pool_get_gram", "vpca_pool_compute_pca",
    "vpca_pool_get_stats", "vpca_debug_tiles", "vpca_debug_plan",
    "vpca_create_projecting", "vpca_get_cross_gram", "vpca_project_pca", "vpca_debug_projection_tiles",
    "vpca_pca_loadings_calls", "vpca_pca_loadings_bed", "vpca_pca_loadings_panels", "vpca_pca_model_terms",
    "vpca_create_scoring", "vpca_score_calls", "vpca_score_bed", "vpca_score_panels", "vpca_score_project",
)


class VpcaError(RuntimeError):
    """Raised for every negative vpca_status (the JNI shim rethrows the same way as RuntimeException)."""

    def __init__(self, code: int, message: str):
        super().__init__(f"vpca {_STATUS_NAMES.get(code, code)}: {message}")
        self.code = code


class IndexOutOfRange(VpcaError, IndexError):
    """Sample index outside [0, N): the reference throws at VariantsPca.scala:59 / :188."""


class VpcaConfig(ctypes.Structure):
    _fields_ = [
        ("struct_size", ctypes.c_uint32),
        ("n_samples", ctypes.c_int32),
        ("device", ctypes.c_int32),
        ("dtype", ctypes.c_int32),
        ("num_pc", ctypes.c_int32),
        ("max_multiplicity", ctypes.c_int32),
        ("partitions_in_flight", ctypes.c_int32),
        ("staging_lanes", ctypes.c_int32),
        ("chunk_variants", ctypes.c_int64),
        ("chunk_nnz", ctypes.c_int64),
        ("stream", ctypes.c_void_p),
        ("d_gram", ctypes.c_void_p),
        ("gram_band_row0", ctypes.c_int32),
        ("gram_band_rows", ctypes.c_int32),
    ]


class VpcaProjection(ctypes.Structure):
    _fields_ = [
        ("struct_size", ctypes.c_uint32),
        ("n_projected", ctypes.c_int32),
        ("sample_rows", ctypes.POINTER(ctypes.c_int32)),
    ]


class VpcaModel(ctypes.Structure):
    _fields_ = [
        ("struct_size", ctypes.c_uint32),
        ("n_fitted", ctypes.c_int32),
        ("k", ctypes.c_int32),
        ("n_variants", ctypes.c_int64),
        ("loadings", ctypes.c_void_p),
        ("carriers", ctypes.c_void_p),
        ("eigenvalues", ctypes.c_void_p),
        ("col_sums", ctypes.c_void_p),
        ("rowsum_dots", ctypes.c_void_p),
        ("matrix_mean", ctypes.c_double),
    ]


class VpcaStats(ctypes.Structure):
    _fields_ = [
        ("variants_accumulated", ctypes.c_int64),
        ("gram_launches", ctypes.c_int64),
        ("kernel_launches", ctypes.c_int64),
        ("h2d_bytes", ctypes.c_int64),
        ("d2h_bytes", ctypes.c_int64),
        ("last_gram_ms", ctypes.c_float),
        ("last_eig_ms", ctypes.c_float),
        ("gram_cta_group", ctypes.c_int32),
        ("gram_resident", ctypes.c_int32),
        ("eig_method", ctypes.c_int32),
        ("eig_iterations", ctypes.c_int32),
    ]


_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libvpca.so"
_lib: Optional[ctypes.CDLL] = None


def library_path() -> Path:
    return Path(os.environ.get("VPCA_LIBRARY", str(LIB_PATH)))


def load_library() -> ctypes.CDLL:
    """dlopen libvpca.so and declare the prototypes.  Raises VpcaError if the library is not built."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not path.exists():
        raise VpcaError(VPCA_ERR_CUDA, f"{path} not found: build it with `python -c 'import __graft_entry__ as g; "
                        "g.build()'` (there is no CPU fallback)")
    L = ctypes.CDLL(str(path))
    vp, i64, i32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32
    L.vpca_version.restype = ctypes.c_int
    L.vpca_version.argtypes = []
    L.vpca_create.restype = ctypes.c_int
    L.vpca_create.argtypes = [ctypes.POINTER(VpcaConfig), ctypes.POINTER(vp)]
    L.vpca_destroy.restype = ctypes.c_int
    L.vpca_destroy.argtypes = [vp]
    L.vpca_last_error.restype = ctypes.c_char_p
    L.vpca_last_error.argtypes = [vp]
    L.vpca_reset.restype = ctypes.c_int
    L.vpca_reset.argtypes = [vp]
    L.vpca_encode_calls.restype = ctypes.c_int
    L.vpca_encode_calls.argtypes = [vp, vp, vp, i64, vp, i64]
    L.vpca_accumulate_calls.restype = ctypes.c_int
    L.vpca_accumulate_calls.argtypes = [vp, i64, vp, vp, i64]
    L.vpca_accumulate_calls_u16.restype = ctypes.c_int
    L.vpca_accumulate_calls_u16.argtypes = [vp, i64, vp, vp, i64]
    L.vpca_hash_keys.restype = ctypes.c_int
    L.vpca_hash_keys.argtypes = [vp, vp, vp, i64, vp]
    L.vpca_join_rows.restype = ctypes.c_int
    L.vpca_join_rows.argtypes = [vp, i32, i32, i64, vp, vp, vp, vp, i64, ctypes.POINTER(i64), ctypes.POINTER(i64)]
    L.vpca_join_size.restype = ctypes.c_int
    L.vpca_join_size.argtypes = [vp, ctypes.POINTER(i64), ctypes.POINTER(i64)]
    L.vpca_join_fetch.restype = ctypes.c_int
    L.vpca_join_fetch.argtypes = [vp, vp, vp]
    L.vpca_accumulate_joined.restype = ctypes.c_int
    L.vpca_accumulate_joined.argtypes = [vp, i64]
    L.vpca_accumulate_bits.restype = ctypes.c_int
    L.vpca_accumulate_bits.argtypes = [vp, i64, vp, i64, i64]
    L.vpca_accumulate_bed.restype = ctypes.c_int
    L.vpca_accumulate_bed.argtypes = [vp, i64, vp, i64, i64, ctypes.c_int32]
    L.vpca_commit.restype = ctypes.c_int
    L.vpca_commit.argtypes = [vp, i64]
    L.vpca_abort.restype = ctypes.c_int
    L.vpca_abort.argtypes = [vp, i64]
    L.vpca_accumulate_dense.restype = ctypes.c_int
    L.vpca_accumulate_dense.argtypes = [vp, vp, i64, i64, ctypes.c_int]
    L.vpca_gram_device_ptr.restype = ctypes.c_int
    L.vpca_gram_device_ptr.argtypes = [vp, ctypes.POINTER(vp)]
    L.vpca_finalize_gram.restype = ctypes.c_int
    L.vpca_finalize_gram.argtypes = [vp]
    L.vpca_get_gram.restype = ctypes.c_int
    L.vpca_get_gram.argtypes = [vp, vp]
    L.vpca_get_partial_gram.restype = ctypes.c_int
    L.vpca_get_partial_gram.argtypes = [vp, vp, ctypes.POINTER(i64)]
    L.vpca_load_partial_gram.restype = ctypes.c_int
    L.vpca_load_partial_gram.argtypes = [vp, vp, i64]
    L.vpca_variant_count.restype = i64
    L.vpca_variant_count.argtypes = [vp]
    L.vpca_synchronize.restype = ctypes.c_int
    L.vpca_synchronize.argtypes = [vp]
    L.vpca_host_alloc.restype = ctypes.c_int
    L.vpca_host_alloc.argtypes = [ctypes.c_size_t, ctypes.POINTER(vp)]
    L.vpca_host_free.restype = ctypes.c_int
    L.vpca_host_free.argtypes = [vp]
    L.vpca_gram_set_peers_local.restype = ctypes.c_int
    L.vpca_gram_set_peers_local.argtypes = [ctypes.POINTER(vp), i32]
    L.vpca_owner_row_bands.restype = ctypes.c_int
    L.vpca_owner_row_bands.argtypes = [i32, i32, ctypes.POINTER(i32)]
    L.vpca_get_gram_band.restype = ctypes.c_int
    L.vpca_get_gram_band.argtypes = [vp, i32, i32, vp]
    L.vpca_pool_create.restype = ctypes.c_int
    L.vpca_pool_create.argtypes = [ctypes.POINTER(VpcaConfig), i32, ctypes.POINTER(i32), ctypes.POINTER(vp)]
    L.vpca_pool_destroy.restype = ctypes.c_int
    L.vpca_pool_destroy.argtypes = [vp]
    L.vpca_pool_size.restype = i32
    L.vpca_pool_size.argtypes = [vp]
    L.vpca_pool_ctx.restype = vp
    L.vpca_pool_ctx.argtypes = [vp, i64]
    L.vpca_pool_last_error.restype = ctypes.c_char_p
    L.vpca_pool_last_error.argtypes = [vp]
    L.vpca_pool_reset.restype = ctypes.c_int
    L.vpca_pool_reset.argtypes = [vp]
    L.vpca_pool_accumulate_calls.restype = ctypes.c_int
    L.vpca_pool_accumulate_calls.argtypes = [vp, i64, vp, vp, i64]
    L.vpca_pool_accumulate_calls_u16.restype = ctypes.c_int
    L.vpca_pool_accumulate_calls_u16.argtypes = [vp, i64, vp, vp, i64]
    L.vpca_pool_accumulate_bits.restype = ctypes.c_int
    L.vpca_pool_accumulate_bits.argtypes = [vp, i64, vp, i64, i64]
    L.vpca_pool_accumulate_bed.restype = ctypes.c_int
    L.vpca_pool_accumulate_bed.argtypes = [vp, i64, vp, i64, i64, i32]
    L.vpca_pool_commit.restype = ctypes.c_int
    L.vpca_pool_commit.argtypes = [vp, i64]
    L.vpca_pool_abort.restype = ctypes.c_int
    L.vpca_pool_abort.argtypes = [vp, i64]
    L.vpca_pool_reduce_and_finalize.restype = ctypes.c_int
    L.vpca_pool_reduce_and_finalize.argtypes = [vp]
    L.vpca_pool_get_gram.restype = ctypes.c_int
    L.vpca_pool_get_gram.argtypes = [vp, vp]
    L.vpca_pool_compute_pca.restype = ctypes.c_int
    L.vpca_pool_compute_pca.argtypes = [vp, i32, vp, vp, ctypes.POINTER(i32)]
    L.vpca_pool_get_stats.restype = ctypes.c_int
    L.vpca_pool_get_stats.argtypes = [vp, ctypes.POINTER(VpcaStats)]
    L.vpca_debug_tiles.restype = ctypes.c_int
    L.vpca_debug_tiles.argtypes = [i32, i32, i32, vp, i32]
    L.vpca_debug_plan.restype = ctypes.c_int
    L.vpca_debug_plan.argtypes = [vp, i32, i32, i32, vp, i32]
    L.vpca_debug_lanczos_profile.restype = ctypes.c_int
    L.vpca_debug_lanczos_profile.argtypes = [vp, vp, i32]
    L.vpca_debug_rebalance.restype = ctypes.c_int
    L.vpca_debug_rebalance.argtypes = [vp, i32, i32, i32, i32, vp, vp, i32]
    L.vpca_set_gram.restype = ctypes.c_int
    L.vpca_set_gram.argtypes = [vp, vp]
    L.vpca_compute_pca.restype = ctypes.c_int
    L.vpca_compute_pca.argtypes = [vp, i32, vp, vp, ctypes.POINTER(i32)]
    L.vpca_get_centered.restype = ctypes.c_int
    L.vpca_get_centered.argtypes = [vp, vp]
    L.vpca_get_tridiagonal.restype = ctypes.c_int
    L.vpca_get_tridiagonal.argtypes = [vp, vp, vp]
    L.vpca_synth_dense_device.restype = ctypes.c_int
    L.vpca_synth_dense_device.argtypes = [vp, ctypes.c_uint64, i64, i64, ctypes.c_int, vp, i64]
    L.vpca_get_stats.restype = ctypes.c_int
    L.vpca_get_stats.argtypes = [vp, ctypes.POINTER(VpcaStats)]
    L.vpca_accumulate_panels.restype = ctypes.c_int
    L.vpca_accumulate_panels.argtypes = [vp, vp, i64, i64]
    L.vpca_synth_panels_device.restype = ctypes.c_int
    L.vpca_synth_panels_device.argtypes = [vp, ctypes.c_uint64, i64, i64, ctypes.c_int, vp, i64]
    L.vpca_gram_export_ipc.restype = ctypes.c_int
    L.vpca_gram_export_ipc.argtypes = [vp, vp]
    L.vpca_gram_set_peers.restype = ctypes.c_int
    L.vpca_gram_set_peers.argtypes = [vp, vp, i32, i32]
    L.vpca_peer_barrier.restype = ctypes.c_int
    L.vpca_peer_barrier.argtypes = [vp]
    L.vpca_gram_set_peer_mode.restype = ctypes.c_int
    L.vpca_gram_set_peer_mode.argtypes = [vp, ctypes.c_int32]
    L.vpca_gram_gather.restype = ctypes.c_int
    L.vpca_gram_gather.argtypes = [vp]
    L.vpca_debug_gram_profile.restype = ctypes.c_int
    L.vpca_debug_gram_profile.argtypes = [vp, vp, i32]
    L.vpca_create_projecting.restype = ctypes.c_int
    L.vpca_create_projecting.argtypes = [ctypes.POINTER(VpcaConfig), ctypes.POINTER(VpcaProjection), ctypes.POINTER(vp)]
    L.vpca_get_cross_gram.restype = ctypes.c_int
    L.vpca_get_cross_gram.argtypes = [vp, vp]
    L.vpca_project_pca.restype = ctypes.c_int
    L.vpca_project_pca.argtypes = [vp, i32, vp]
    L.vpca_debug_projection_tiles.restype = ctypes.c_int
    L.vpca_debug_projection_tiles.argtypes = [i32, i32, i32, i32, vp, i32]
    L.vpca_pca_loadings_calls.restype = ctypes.c_int
    L.vpca_pca_loadings_calls.argtypes = [vp, i32, vp, vp, i64, vp, vp]
    L.vpca_pca_loadings_bed.restype = ctypes.c_int
    L.vpca_pca_loadings_bed.argtypes = [vp, i32, vp, i64, i64, i32, vp, vp]
    L.vpca_pca_loadings_panels.restype = ctypes.c_int
    L.vpca_pca_loadings_panels.argtypes = [vp, i32, vp, i64, i64, vp, vp]
    L.vpca_pca_model_terms.restype = ctypes.c_int
    L.vpca_pca_model_terms.argtypes = [vp, i32, vp, vp, vp, vp]
    L.vpca_create_scoring.restype = ctypes.c_int
    L.vpca_create_scoring.argtypes = [ctypes.POINTER(VpcaConfig), ctypes.POINTER(VpcaModel), ctypes.POINTER(vp)]
    L.vpca_score_calls.restype = ctypes.c_int
    L.vpca_score_calls.argtypes = [vp, i64, vp, vp, i64, vp]
    L.vpca_score_bed.restype = ctypes.c_int
    L.vpca_score_bed.argtypes = [vp, i64, vp, i64, i64, i32, vp]
    L.vpca_score_panels.restype = ctypes.c_int
    L.vpca_score_panels.argtypes = [vp, vp, i64, i64, vp]
    L.vpca_score_project.restype = ctypes.c_int
    L.vpca_score_project.argtypes = [vp, i32, vp, ctypes.POINTER(i64)]
    _lib = L
    return L


def _host_ptr(a: np.ndarray) -> int:
    return a.ctypes.data


class NativePca:
    """One GPU's VariantsPca state.  Method names follow the JNI class of INTEGRATION.md 1:1."""

    def __init__(self, n_samples: int, device: int = 0, dtype: int = DTYPE_I8, num_pc: int = 2,
                 max_multiplicity: int = 2, partitions_in_flight: int = 4, chunk_variants: int = 0,
                 chunk_nnz: int = 0, stream: int = 0, d_gram: int = 0, staging_lanes: int = 0,
                 gram_band: Optional[Tuple[int, int]] = None, n_projected: int = 0, sample_rows=None, model=None):
        """n_projected > 0 (or a sample_rows map): a projecting context (vpca_create_projecting) -- n_samples fitted
        samples plus n_projected ones placed on the fitted PCs by projectPca.  sample_rows: input sample position ->
        row of the context (fitted rows first), None = the last n_projected inputs are the projected ones.
        model: a scoring context (vpca_create_scoring) for n_samples study samples -- an object with the fields of
        vpca_model (n_fitted, loadings (V, k), carriers (V,), eigenvalues, col_sums, rowsum_dots (k,), matrix_mean),
        such as model.PcaModel; it has no Gram, only the score* methods."""
        self._lib = load_library()
        self.n = int(n_samples)
        self.n_projected = int(n_projected)
        self.rows = self.n + self.n_projected   # rows of the genotype tiles and of the Gram buffer
        self.dtype = int(dtype)
        self.elem_bits = {DTYPE_I8: 8, DTYPE_BF16: 16, DTYPE_E2M1: 4}[self.dtype]
        self.elem_bytes = self.elem_bits / 8
        self.max_multiplicity = int(max_multiplicity) if max_multiplicity > 0 else 2
        row0, rows = gram_band if gram_band is not None else (0, 0)
        cfg = VpcaConfig(ctypes.sizeof(VpcaConfig), n_samples, device, dtype, num_pc, max_multiplicity,
                         partitions_in_flight, staging_lanes, chunk_variants, chunk_nnz, stream or None, d_gram or None,
                         row0, rows)
        handle = ctypes.c_void_p()
        self.model_k = 0
        if model is not None:
            L = np.ascontiguousarray(model.loadings, dtype=np.float64)
            n_var, k = L.shape
            cnt = np.ascontiguousarray(model.carriers, dtype=np.int32)
            terms = [np.ascontiguousarray(getattr(model, f), dtype=np.float64)
                     for f in ("eigenvalues", "col_sums", "rowsum_dots")]
            if cnt.shape != (n_var,) or any(t.shape != (k,) for t in terms):
                raise VpcaError(VPCA_ERR_BAD_ARG, "model: carriers must have V entries and the terms k")
            vm = VpcaModel(ctypes.sizeof(VpcaModel), int(model.n_fitted), k, n_var, _host_ptr(L) if n_var else None,
                           _host_ptr(cnt) if n_var else None, *[_host_ptr(t) for t in terms], float(model.matrix_mean))
            rc = self._lib.vpca_create_scoring(ctypes.byref(cfg), ctypes.byref(vm), ctypes.byref(handle))
            self.model_k = k
        elif self.n_projected > 0 or sample_rows is not None:
            rows_map = None
            if sample_rows is not None:
                rows_map = np.ascontiguousarray(sample_rows, dtype=np.int32)
                if rows_map.shape != (self.rows,):
                    raise VpcaError(VPCA_ERR_BAD_ARG, f"sample_rows must have n_samples + n_projected = {self.rows} entries")
            proj = VpcaProjection(ctypes.sizeof(VpcaProjection), self.n_projected,
                                  rows_map.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)) if rows_map is not None else None)
            rc = self._lib.vpca_create_projecting(ctypes.byref(cfg), ctypes.byref(proj), ctypes.byref(handle))
        else:
            rc = self._lib.vpca_create(ctypes.byref(cfg), ctypes.byref(handle))
        self._h = handle if rc == VPCA_OK else None
        if rc != VPCA_OK:
            self._raise(rc, None)

    # -- error plumbing ------------------------------------------------------------------------
    def _raise(self, rc: int, handle):
        msg = self._lib.vpca_last_error(handle).decode("utf-8", "replace")
        if rc == VPCA_ERR_INDEX_OUT_OF_RANGE:
            raise IndexOutOfRange(rc, msg)
        raise VpcaError(rc, msg)

    def _check(self, rc: int):
        if rc != VPCA_OK:
            self._raise(rc, self._h)

    def close(self):
        if getattr(self, "_h", None) is not None:
            self._lib.vpca_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- API -------------------------------------------------------------------------------------
    def reset(self):
        self._check(self._lib.vpca_reset(self._h))

    @staticmethod
    def _csr(offsets, sample_idx) -> Tuple[np.ndarray, np.ndarray]:
        off = np.ascontiguousarray(offsets, dtype=np.int64)
        idx = np.ascontiguousarray(sample_idx, dtype=np.int32)
        if off.ndim != 1 or len(off) < 1:
            raise VpcaError(VPCA_ERR_BAD_ARG, "offsets must be a 1-D array with nv+1 entries")
        return off, idx

    def encodeCalls(self, offsets, sample_idx) -> np.ndarray:
        """Device encode only (CSR rows -> dense sample-major tile), copied back: shape (n, nv)."""
        off, idx = self._csr(offsets, sample_idx)
        nv = len(off) - 1
        if self.elem_bits == 4:                      # packed: (n, ld / 2) bytes, ld a multiple of 128 cells
            ld = max(128, ((nv + 127) // 128) * 128)
            out = np.zeros((self.rows, ld // 2), dtype=np.uint8)
            self._check(self._lib.vpca_encode_calls(self._h, _host_ptr(off), _host_ptr(idx) if len(idx) else None, nv,
                                                    _host_ptr(out), ld))
            return out
        out = np.zeros((self.rows, max(nv, 1)), dtype=np.int8 if self.elem_bits == 8 else np.uint16)
        self._check(self._lib.vpca_encode_calls(self._h, _host_ptr(off), _host_ptr(idx) if len(idx) else None, nv,
                                                _host_ptr(out), out.shape[1]))
        return out[:, :nv]

    def accumulateCalls(self, partition_id: int, offsets, sample_idx):
        off, idx = self._csr(offsets, sample_idx)
        self._check(self._lib.vpca_accumulate_calls(self._h, int(partition_id), _host_ptr(off),
                                                    _host_ptr(idx) if len(idx) else None, len(off) - 1))

    # -- multi-dataset keying on the device (VariantsPca.scala:62-78, :115-148) --------------------------------------
    @staticmethod
    def _keys(keys):
        """list of bytes -> (payload uint8, key_offsets int64)"""
        lens = np.fromiter((len(k) for k in keys), dtype=np.int64, count=len(keys))
        koff = np.zeros(len(keys) + 1, dtype=np.int64)
        np.cumsum(lens, out=koff[1:])
        payload = np.frombuffer(b"".join(keys), dtype=np.uint8) if len(keys) else np.zeros(0, np.uint8)
        return np.ascontiguousarray(payload), koff

    def hashKeys(self, keys) -> np.ndarray:
        """MurmurHash3_x64_128 of every byte string in `keys`, computed on the GPU: (len(keys), 2) uint64 (h1, h2);
        `bytes(row).hex()` of a little-endian row is Guava's HashCode.toString (vpca_hash_keys)."""
        payload, koff = self._keys(keys)
        out = np.zeros((len(keys), 2), dtype=np.uint64)
        self._check(self._lib.vpca_hash_keys(self._h, _host_ptr(payload) if len(payload) else None, _host_ptr(koff),
                                             len(keys), _host_ptr(out) if len(keys) else None))
        return out

    def joinRows(self, mode: int, keys, offsets, sample_idx, n_left: int = 0, variant_set_count: int = 2):
        """Join (mode JOIN: rows [0, n_left) x rows [n_left, ...)) or merge (mode MERGE) of the rows of several datasets on
        their variant keys, on the GPU; the joined rows stay there (accumulateJoined / joinFetch).  Returns (rows, calls)."""
        payload, koff = self._keys(keys)
        off, idx = self._csr(offsets, sample_idx)
        if len(off) - 1 != len(keys):
            raise VpcaError(VPCA_ERR_BAD_ARG, "one key per row")
        rows, nnz = ctypes.c_int64(0), ctypes.c_int64(0)
        self._check(self._lib.vpca_join_rows(self._h, int(mode), int(variant_set_count), int(n_left),
                                             _host_ptr(payload) if len(payload) else None, _host_ptr(koff), _host_ptr(off),
                                             _host_ptr(idx) if len(idx) else None, len(keys), ctypes.byref(rows),
                                             ctypes.byref(nnz)))
        return int(rows.value), int(nnz.value)

    def joinSize(self):
        """(rows, calls) of the joined rows the context retains (vpca_join_size)."""
        rows, nnz = ctypes.c_int64(0), ctypes.c_int64(0)
        self._check(self._lib.vpca_join_size(self._h, ctypes.byref(rows), ctypes.byref(nnz)))
        return int(rows.value), int(nnz.value)

    def joinFetch(self, rows: int, nnz: int):
        """The joined rows of the last joinRows as a host CSR (offsets int64, sample indices int32)."""
        off = np.zeros(rows + 1, dtype=np.int64)
        idx = np.zeros(max(nnz, 1), dtype=np.int32)
        self._check(self._lib.vpca_join_fetch(self._h, _host_ptr(off), _host_ptr(idx)))
        return off, idx[:nnz]

    def lanczosProfile(self) -> np.ndarray:
        """(steps, 8) int64 ns timestamps of block 0 of the persistent Lanczos kernel (VPCA_LZ_PROF=1)."""
        out = np.zeros((32, 8), dtype=np.int64)
        cnt = self._lib.vpca_debug_lanczos_profile(self._h, _host_ptr(out), 32)
        if cnt < 0:
            self._check(cnt)
        return out[:cnt]

    def accumulateJoined(self, partition_id: int):
        """Encode + Gram of the joined rows of the last joinRows, straight from device memory (vpca_accumulate_joined)."""
        self._check(self._lib.vpca_accumulate_joined(self._h, int(partition_id)))

    def accumulateCallsRaw(self, partition_id: int, off_ptr: int, idx_ptr: int, nv: int, idx_bytes: int = 4):
        """Same, from raw host addresses (e.g. pinned torch tensors) -- no copies on the Python side.
        idx_bytes = 2: the indices are uint16 (vpca_accumulate_calls_u16)."""
        fn = self._lib.vpca_accumulate_calls if idx_bytes == 4 else self._lib.vpca_accumulate_calls_u16
        self._check(fn(self._h, int(partition_id), off_ptr, idx_ptr, int(nv)))

    def accumulateBits(self, partition_id: int, bits: np.ndarray):
        """bits: (nv, stride) uint8, bit s (LSB first) of row v = sample s carries variant v."""
        b = np.ascontiguousarray(bits, dtype=np.uint8)
        if b.ndim != 2:
            raise VpcaError(VPCA_ERR_BAD_ARG, "bits must be (nv, stride_bytes)")
        self._check(self._lib.vpca_accumulate_bits(self._h, int(partition_id), _host_ptr(b), b.shape[0], b.shape[1]))

    def accumulateBed(self, partition_id: int, rows: np.ndarray, counted_allele: int = 1):
        """rows: (nv, stride) uint8 PLINK .bed rows (2 bits per sample: 00 hom A1, 01 missing, 10 het, 11 hom A2);
        counted_allele 1: carriers of A1, 2: carriers of A2 (plink.py)."""
        b = np.ascontiguousarray(rows, dtype=np.uint8)
        if b.ndim != 2:
            raise VpcaError(VPCA_ERR_BAD_ARG, "rows must be (nv, stride_bytes)")
        self._check(self._lib.vpca_accumulate_bed(self._h, int(partition_id), _host_ptr(b), b.shape[0], b.shape[1],
                                                  int(counted_allele)))

    def accumulateBitsRaw(self, partition_id: int, ptr: int, nv: int, stride_bytes: int):
        self._check(self._lib.vpca_accumulate_bits(self._h, int(partition_id), ptr, int(nv), int(stride_bytes)))

    def accumulateCalls16(self, partition_id: int, offsets, sample_idx):
        off = np.ascontiguousarray(offsets, dtype=np.int64)
        idx = np.ascontiguousarray(sample_idx, dtype=np.uint16)
        self._check(self._lib.vpca_accumulate_calls_u16(self._h, int(partition_id), _host_ptr(off),
                                                        _host_ptr(idx) if len(idx) else None, len(off) - 1))

    def commit(self, partition_id: int):
        self._check(self._lib.vpca_commit(self._h, int(partition_id)))

    def abort(self, partition_id: int):
        self._check(self._lib.vpca_abort(self._h, int(partition_id)))

    def accumulateDense(self, x: np.ndarray, nv: Optional[int] = None):
        """Host dense tile, shape (n, nv), int8 (or uint16 bf16 bits); for DTYPE_E2M1 packed uint8 of shape
        (n, ld / 2) with ld % 128 == 0, `nv` valid cells per row and zero cells after them."""
        x = np.asarray(x)
        if self.elem_bits == 4:
            if x.dtype != np.uint8 or x.ndim != 2 or x.shape[0] != self.rows or (x.shape[1] * 2) % 128:
                raise VpcaError(VPCA_ERR_BAD_ARG, f"packed tile must be ({self.rows}, ld/2) uint8 with ld % 128 == 0")
            x = np.ascontiguousarray(x)
            ld = x.shape[1] * 2
            self._check(self._lib.vpca_accumulate_dense(self._h, _host_ptr(x), ld if nv is None else int(nv), ld, 0))
            return
        want = np.int8 if self.elem_bits == 8 else np.uint16
        if x.dtype != want or x.ndim != 2 or x.shape[0] != self.rows:
            raise VpcaError(VPCA_ERR_BAD_ARG, f"dense tile must be ({self.rows}, nv) {np.dtype(want).name}")
        if not x.flags.c_contiguous:
            x = np.ascontiguousarray(x)
        self._check(self._lib.vpca_accumulate_dense(self._h, _host_ptr(x), x.shape[1], x.shape[1], 0))

    def accumulateDenseDevice(self, d_ptr: int, nv: int, ld: int):
        self._check(self._lib.vpca_accumulate_dense(self._h, d_ptr, int(nv), int(ld), 1))

    def accumulatePanels(self, d_ptr: int, nv: int, panel_variants: int):
        """Device-resident cohort in panel layout (see vpca.h): one Gram launch over all nv variants."""
        self._check(self._lib.vpca_accumulate_panels(self._h, d_ptr, int(nv), int(panel_variants)))

    def synthPanelsDevice(self, seed: int, v0: int, nv: int, mode: int, d_ptr: int, panel_variants: int):
        self._check(self._lib.vpca_synth_panels_device(self._h, ctypes.c_uint64(seed), int(v0), int(nv), int(mode),
                                                       d_ptr, int(panel_variants)))

    def panelBytes(self, nv: int, panel_variants: int) -> int:
        npanels = (int(nv) + panel_variants - 1) // panel_variants
        return npanels * self.rows * panel_variants * self.elem_bits // 8

    def gramDevicePtr(self) -> int:
        p = ctypes.c_void_p()
        self._check(self._lib.vpca_gram_device_ptr(self._h, ctypes.byref(p)))
        return int(p.value)

    def exportIpcHandle(self) -> bytes:
        buf = ctypes.create_string_buffer(64)
        self._check(self._lib.vpca_gram_export_ipc(self._h, buf))
        return buf.raw

    def setPeers(self, handles, rank: int, mode: str = "replicate"):
        """handles: list of 64-byte handles of all ranks, in rank order.  mode: "replicate" (every flush into every
        rank's Gram) or "owner_rows" (reduce-scatter by Gram row bands; finish a pass with gatherGram())."""
        blob = ctypes.create_string_buffer(b"".join(handles), 64 * len(handles))
        self._check(self._lib.vpca_gram_set_peers(self._h, blob, len(handles), int(rank)))
        self._check(self._lib.vpca_gram_set_peer_mode(self._h, {"replicate": 0, "owner_rows": 1}[mode]))

    def gatherGram(self):
        """Closing step of a fused pass: all-rank barrier (+ pull of the other ranks' row bands in owner_rows mode)."""
        self._check(self._lib.vpca_gram_gather(self._h))

    def peerBarrier(self):
        self._check(self._lib.vpca_peer_barrier(self._h))

    def finalizeGram(self):
        self._check(self._lib.vpca_finalize_gram(self._h))

    def getGram(self) -> np.ndarray:
        out = np.empty((self.n, self.n), dtype=np.int32)
        self._check(self._lib.vpca_get_gram(self._h, _host_ptr(out)))
        return out

    def partialGram(self, with_count: bool = False):
        """The accumulated (not yet finalized) Gram: lower triangle meaningful.  Checkpoint payload (with_count: also
        the number of variants the counts stand for, which a resume hands back to loadPartialGram).  Projecting
        contexts: (n + n_projected, n), the cross block below the fitted Gram."""
        out = np.empty((self.rows, self.n), dtype=np.int32)
        nv = ctypes.c_int64(0)
        self._check(self._lib.vpca_get_partial_gram(self._h, _host_ptr(out), ctypes.byref(nv)))
        return (out, int(nv.value)) if with_count else out

    def loadPartialGram(self, gram: np.ndarray, variants_in_gram: int):
        """Restore a checkpointed partial Gram; accumulation continues on top of it (and keeps counting against the
        int32 bound of a similarity count from `variants_in_gram`)."""
        g = np.ascontiguousarray(gram, dtype=np.int32)
        if g.shape != (self.rows, self.n):
            raise VpcaError(VPCA_ERR_BAD_ARG, "gram must be (n + n_projected, n)")
        self._check(self._lib.vpca_load_partial_gram(self._h, _host_ptr(g), int(variants_in_gram)))

    def variantCount(self) -> int:
        v = int(self._lib.vpca_variant_count(self._h))
        if v < 0:
            self._raise(v, self._h)
        return v

    def synchronize(self):
        self._check(self._lib.vpca_synchronize(self._h))

    def gramBand(self, row0: int, rows: int) -> np.ndarray:
        """Rows [row0, row0 + rows) of the Gram as this context stores them (band-only contexts: their own band)."""
        out = np.empty((rows, self.n), dtype=np.int32)
        self._check(self._lib.vpca_get_gram_band(self._h, int(row0), int(rows), _host_ptr(out)))
        return out

    def setGram(self, gram: np.ndarray):
        g = np.ascontiguousarray(gram, dtype=np.int32)
        if g.shape != (self.n, self.n):
            raise VpcaError(VPCA_ERR_BAD_ARG, "gram must be (n, n)")
        self._check(self._lib.vpca_set_gram(self._h, _host_ptr(g)))

    def computePca(self, k: int = 2):
        """-> (vecs (n, k) with column c = PC c, evals (k,), nonZeroRows).  `vecs.T.ravel()` is the
        column-major array ``pca.toArray`` of VariantsPca.scala:227."""
        flat = np.empty(self.n * k, dtype=np.float64)
        evals = np.empty(k, dtype=np.float64)
        nz = ctypes.c_int32(0)
        self._check(self._lib.vpca_compute_pca(self._h, int(k), _host_ptr(flat), _host_ptr(evals), ctypes.byref(nz)))
        return flat.reshape(k, self.n).T.copy(), evals, int(nz.value)

    def crossGram(self) -> np.ndarray:
        """(n_projected, n) int32: variants each projected sample shares with each fitted one (after finalizeGram)."""
        out = np.empty((self.n_projected, self.n), dtype=np.int32)
        self._check(self._lib.vpca_get_cross_gram(self._h, _host_ptr(out)))
        return out

    def projectPca(self, k: int = 2) -> np.ndarray:
        """(n_projected, k) float64: coordinates of the projected samples on the first k PCs of the last computePca."""
        flat = np.empty(max(self.n_projected * k, 1), dtype=np.float64)
        self._check(self._lib.vpca_project_pca(self._h, int(k), _host_ptr(flat)))
        return flat[:self.n_projected * k].reshape(k, self.n_projected).T.copy()

    # -- saved model (DESIGN.md 3.7): loadings of a fitted context ... ----------------------------------------------
    def pcaLoadingsCalls(self, k: int, offsets, sample_idx):
        """Loadings of the rows of an accumulate call on the first k PCs of the last computePca: (L (nv, k) float64,
        carriers (nv,) int32), one row per input variant."""
        off, idx = self._csr(offsets, sample_idx)
        nv = len(off) - 1
        L, cnt = np.empty((nv, k), np.float64), np.empty(nv, np.int32)
        self._check(self._lib.vpca_pca_loadings_calls(self._h, int(k), _host_ptr(off), _host_ptr(idx) if len(idx) else None,
                                                      nv, _host_ptr(L), _host_ptr(cnt)))
        return L, cnt

    def pcaLoadingsBed(self, k: int, rows: np.ndarray, counted_allele: int = 1):
        b = np.ascontiguousarray(rows, dtype=np.uint8)
        if b.ndim != 2:
            raise VpcaError(VPCA_ERR_BAD_ARG, "rows must be (nv, stride_bytes)")
        L, cnt = np.empty((b.shape[0], k), np.float64), np.empty(b.shape[0], np.int32)
        self._check(self._lib.vpca_pca_loadings_bed(self._h, int(k), _host_ptr(b), b.shape[0], b.shape[1],
                                                    int(counted_allele), _host_ptr(L), _host_ptr(cnt)))
        return L, cnt

    def pcaLoadingsPanels(self, k: int, d_ptr: int, nv: int, panel_variants: int):
        L, cnt = np.empty((nv, k), np.float64), np.empty(nv, np.int32)
        self._check(self._lib.vpca_pca_loadings_panels(self._h, int(k), d_ptr, int(nv), int(panel_variants), _host_ptr(L),
                                                       _host_ptr(cnt)))
        return L, cnt

    def pcaModelTerms(self, k: int) -> dict:
        """eigenvalues, col_sums (a), rowsum_dots (b) and matrix_mean of the last computePca."""
        ev, a, b = (np.empty(k, np.float64) for _ in range(3))
        mm = np.empty(1, np.float64)
        self._check(self._lib.vpca_pca_model_terms(self._h, int(k), _host_ptr(ev), _host_ptr(a), _host_ptr(b), _host_ptr(mm)))
        return dict(eigenvalues=ev, col_sums=a, rowsum_dots=b, matrix_mean=float(mm[0]))

    # -- ... and scoring of a study against it (contexts made with model=) -------------------------------------------
    @staticmethod
    def _model_rows(model_rows, nv: int) -> np.ndarray:
        r = np.ascontiguousarray(model_rows, dtype=np.int32)
        if r.shape != (nv,):
            raise VpcaError(VPCA_ERR_BAD_ARG, f"model_rows must have one entry per variant ({nv})")
        return r

    def scoreCalls(self, partition_id: int, offsets, sample_idx, model_rows):
        off, idx = self._csr(offsets, sample_idx)
        r = self._model_rows(model_rows, len(off) - 1)
        self._check(self._lib.vpca_score_calls(self._h, int(partition_id), _host_ptr(off), _host_ptr(idx) if len(idx) else None,
                                               len(off) - 1, _host_ptr(r) if len(r) else None))

    def scoreBed(self, partition_id: int, rows: np.ndarray, model_rows, counted_allele: int = 1):
        b = np.ascontiguousarray(rows, dtype=np.uint8)
        if b.ndim != 2:
            raise VpcaError(VPCA_ERR_BAD_ARG, "rows must be (nv, stride_bytes)")
        r = self._model_rows(model_rows, b.shape[0])
        self._check(self._lib.vpca_score_bed(self._h, int(partition_id), _host_ptr(b), b.shape[0], b.shape[1],
                                             int(counted_allele), _host_ptr(r) if len(r) else None))

    def scorePanels(self, d_ptr: int, nv: int, panel_variants: int, model_rows):
        r = self._model_rows(model_rows, nv)
        self._check(self._lib.vpca_score_panels(self._h, d_ptr, int(nv), int(panel_variants), _host_ptr(r) if len(r) else None))

    def scoreProject(self, k: int = 2):
        """-> (y (n_samples, k) float64, matched variants): the study samples on the first k PCs of the model."""
        flat = np.empty(self.n * k, dtype=np.float64)
        matched = ctypes.c_int64(0)
        self._check(self._lib.vpca_score_project(self._h, int(k), _host_ptr(flat), ctypes.byref(matched)))
        return flat.reshape(k, self.n).T.copy(), int(matched.value)

    def getCentered(self) -> np.ndarray:
        out = np.empty((self.n, self.n), dtype=np.float64)
        self._check(self._lib.vpca_get_centered(self._h, _host_ptr(out)))
        return out

    def getTridiagonal(self):
        d = np.empty(self.n, dtype=np.float64)
        e = np.empty(self.n - 1, dtype=np.float64)
        self._check(self._lib.vpca_get_tridiagonal(self._h, _host_ptr(d), _host_ptr(e)))
        return d, e

    def synthDenseDevice(self, seed: int, v0: int, nv: int, mode: int, d_ptr: int, ld: int):
        self._check(self._lib.vpca_synth_dense_device(self._h, ctypes.c_uint64(seed), int(v0), int(nv), int(mode),
                                                      d_ptr, int(ld)))

    def gramProfile(self, max_ctas: int = 1024) -> np.ndarray:
        """(ctas, 4) int64 ns timestamps of the last Gram launch (needs VPCA_GRAM_PROF=1 at first launch)."""
        out = np.zeros((max_ctas, 4), dtype=np.int64)
        rc = self._lib.vpca_debug_gram_profile(self._h, _host_ptr(out), max_ctas)
        if rc < 0:
            self._raise(rc, self._h)
        return out[:rc]

    def stats(self) -> dict:
        st = VpcaStats()
        self._check(self._lib.vpca_get_stats(self._h, ctypes.byref(st)))
        return {name: getattr(st, name) for name, _ in VpcaStats._fields_}


def debugTiles(n_samples: int, cta_group: int = 2, exact: bool = True) -> np.ndarray:
    """(tiles, 8) int32: the Gram kernel's tile list for n_samples (host-only, no GPU needed; see vpca_debug_tiles)."""
    L = load_library()
    cnt = L.vpca_debug_tiles(int(n_samples), int(cta_group), 1 if exact else 0, None, 0)
    if cnt < 0:
        raise VpcaError(cnt, L.vpca_last_error(None).decode("utf-8", "replace"))
    out = np.zeros((cnt, 8), dtype=np.int32)
    L.vpca_debug_tiles(int(n_samples), int(cta_group), 1 if exact else 0, _host_ptr(out), cnt)
    return out


def debugPlan(tiles: np.ndarray, workers: int, kb_window: int) -> np.ndarray:
    """(pieces, 6) int32 {worker, tile, kb_lo, kb_hi, tmem_col, tmem_cols_of_worker} of one window (vpca_debug_plan)."""
    L = load_library()
    t = np.ascontiguousarray(tiles, dtype=np.int32)
    cap = 8 * int(workers) + 8
    out = np.zeros((cap, 6), dtype=np.int32)
    cnt = L.vpca_debug_plan(_host_ptr(t), len(t), int(workers), int(kb_window), _host_ptr(out), cap)
    if cnt < 0:
        raise VpcaError(VPCA_ERR_STATE, L.vpca_last_error(None).decode("utf-8", "replace"))
    return out[:cnt]


def debugProjectionTiles(n_fit: int, n_total: int, cta_group: int, mxf4: bool) -> np.ndarray:
    """Tiles of a projecting context (vpca_debug_projection_tiles), (tiles, 8) int32 like debugTiles."""
    L = load_library()
    cnt = L.vpca_debug_projection_tiles(int(n_fit), int(n_total), int(cta_group), 1 if mxf4 else 0, None, 0)
    if cnt < 0:
        raise VpcaError(cnt, L.vpca_last_error(None).decode("utf-8", "replace"))
    out = np.zeros((cnt, 8), dtype=np.int32)
    L.vpca_debug_projection_tiles(int(n_fit), int(n_total), int(cta_group), 1 if mxf4 else 0, _host_ptr(out), cnt)
    return out


def debugBandTiles(n_samples: int, cta_group: int, row0: int, rows: int) -> np.ndarray:
    """Tiles of an owner-computes band context (vpca_debug_band_tiles), (tiles, 8) int32 like debugTiles."""
    L = load_library()
    L.vpca_debug_band_tiles.restype = ctypes.c_int
    L.vpca_debug_band_tiles.argtypes = [ctypes.c_int32] * 4 + [ctypes.c_void_p, ctypes.c_int32]
    cnt = L.vpca_debug_band_tiles(int(n_samples), int(cta_group), int(row0), int(rows), None, 0)
    if cnt < 0:
        raise VpcaError(cnt, L.vpca_last_error(None).decode("utf-8", "replace"))
    out = np.zeros((cnt, 8), dtype=np.int32)
    L.vpca_debug_band_tiles(int(n_samples), int(cta_group), int(row0), int(rows), _host_ptr(out), cnt)
    return out


def gramSourceFingerprint() -> str:
    """sha256 (16 hex digits) of csrc/gram_sm100.cu with comments and whitespace removed: what an ncu capture of the Gram
    kernel is tied to (profiles/r2_gram_traffic.json) -- editing a comment does not orphan a capture, editing code does."""
    import hashlib
    import re
    src = (Path(__file__).resolve().parent / "csrc" / "gram_sm100.cu").read_text()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    src = re.sub(r"//[^\n]*", "", src)
    src = re.sub(r"\s+", "", src)
    return hashlib.sha256(src.encode()).hexdigest()[:16]


def maxClusters(device: int, cluster_size: int) -> int:
    """Clusters of `cluster_size` Gram-kernel CTAs the device holds at once (vpca_debug_max_clusters)."""
    L = load_library()
    L.vpca_debug_max_clusters.restype = ctypes.c_int
    L.vpca_debug_max_clusters.argtypes = [ctypes.c_int32, ctypes.c_int32]
    c = L.vpca_debug_max_clusters(int(device), int(cluster_size))
    if c < 0:
        raise VpcaError(c, L.vpca_last_error(None).decode("utf-8", "replace"))
    return c


def debugRebalance(tiles: np.ndarray, workers: int, kb_window: int, cum: np.ndarray, col_limit: int = 512):
    """The rebalancer's repair of a candidate split (vpca_debug_rebalance): returns (repaired cum, pieces like debugPlan)."""
    L = load_library()
    t = np.ascontiguousarray(tiles, dtype=np.int32)
    c = np.ascontiguousarray(cum, dtype=np.float64).copy()
    assert c.shape == (workers + 1,)
    cap = 8 * int(workers) + 8
    out = np.zeros((cap, 6), dtype=np.int32)
    cnt = L.vpca_debug_rebalance(_host_ptr(t), len(t), int(workers), int(kb_window), int(col_limit), _host_ptr(c),
                                 _host_ptr(out), cap)
    if cnt < 0:
        raise VpcaError(cnt, L.vpca_last_error(None).decode("utf-8", "replace"))
    return c, out[:cnt]


def ownerRowBands(n_samples: int, world: int) -> list:
    """Row bands of VPCA_PEER_OWNER_ROWS: [(row0, rows)] per rank (vpca_owner_row_bands)."""
    L = load_library()
    ends = (ctypes.c_int32 * world)()
    rc = L.vpca_owner_row_bands(int(n_samples), int(world), ends)
    if rc != VPCA_OK:
        raise VpcaError(rc, L.vpca_last_error(None).decode("utf-8", "replace"))
    out, prev = [], 0
    for q in range(world):
        out.append((prev, int(ends[q]) - prev))
        prev = int(ends[q])
    return out


def setPeersLocal(contexts, mode: str = "owner_rows"):
    """Wire NativePca objects that live in THIS process (any mix of devices) for the fused reduce
    (vpca_gram_set_peers_local); contexts[r] becomes rank r."""
    L = load_library()
    arr = (ctypes.c_void_p * len(contexts))(*[c._h.value for c in contexts])
    rc = L.vpca_gram_set_peers_local(arr, len(contexts))
    if rc != VPCA_OK:
        raise VpcaError(rc, L.vpca_last_error(None).decode("utf-8", "replace"))
    for c in contexts:
        c._check(L.vpca_gram_set_peer_mode(c._h, {"replicate": 0, "owner_rows": 1}[mode]))


class NativePcaPool:
    """One process driving all GPUs of the box: the ctypes twin of the JNI class ``NativePcaPool``
    (spark_examples_b200/jvm/NativePcaPool.scala).  Partition p is served by GPU p % n_gpus; every method except
    reset / reduceAndFinalize / getGram / computePca may be called from many threads at once."""

    def __init__(self, n_samples: int, n_gpus: int, devices=None, dtype: int = DTYPE_I8, num_pc: int = 2,
                 max_multiplicity: int = 2, partitions_in_flight: int = 4, staging_lanes: int = 0,
                 chunk_variants: int = 0, chunk_nnz: int = 0):
        self._lib = load_library()
        self.n = int(n_samples)
        cfg = VpcaConfig(ctypes.sizeof(VpcaConfig), n_samples, 0, dtype, num_pc, max_multiplicity, partitions_in_flight,
                         staging_lanes, chunk_variants, chunk_nnz, None, None, 0, 0)
        devs = None
        if devices is not None:
            devs = (ctypes.c_int32 * n_gpus)(*[int(d) for d in devices])
        h = ctypes.c_void_p()
        rc = self._lib.vpca_pool_create(ctypes.byref(cfg), int(n_gpus), devs, ctypes.byref(h))
        self._h = h if rc == VPCA_OK else None
        if rc != VPCA_OK:
            self._raise(rc)

    def _raise(self, rc: int):
        msg = self._lib.vpca_pool_last_error(self._h).decode("utf-8", "replace")
        if rc == VPCA_ERR_INDEX_OUT_OF_RANGE:
            raise IndexOutOfRange(rc, msg)
        raise VpcaError(rc, msg)

    def _check(self, rc: int):
        if rc != VPCA_OK:
            self._raise(rc)

    def close(self):
        if getattr(self, "_h", None) is not None:
            self._lib.vpca_pool_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    @property
    def size(self) -> int:
        return int(self._lib.vpca_pool_size(self._h))

    def reset(self):
        self._check(self._lib.vpca_pool_reset(self._h))

    def accumulateCalls(self, partition_id: int, offsets, sample_idx):
        off, idx = NativePca._csr(offsets, sample_idx)
        self._check(self._lib.vpca_pool_accumulate_calls(self._h, int(partition_id), _host_ptr(off),
                                                         _host_ptr(idx) if len(idx) else None, len(off) - 1))

    def accumulateCalls16(self, partition_id: int, offsets, sample_idx):
        off = np.ascontiguousarray(offsets, dtype=np.int64)
        idx = np.ascontiguousarray(sample_idx, dtype=np.uint16)
        self._check(self._lib.vpca_pool_accumulate_calls_u16(self._h, int(partition_id), _host_ptr(off),
                                                             _host_ptr(idx) if len(idx) else None, len(off) - 1))

    def accumulateBits(self, partition_id: int, bits: np.ndarray):
        b = np.ascontiguousarray(bits, dtype=np.uint8)
        self._check(self._lib.vpca_pool_accumulate_bits(self._h, int(partition_id), _host_ptr(b), b.shape[0], b.shape[1]))

    def accumulateBed(self, partition_id: int, rows: np.ndarray, counted_allele: int = 1):
        b = np.ascontiguousarray(rows, dtype=np.uint8)
        self._check(self._lib.vpca_pool_accumulate_bed(self._h, int(partition_id), _host_ptr(b), b.shape[0], b.shape[1],
                                                       int(counted_allele)))

    def commit(self, partition_id: int):
        self._check(self._lib.vpca_pool_commit(self._h, int(partition_id)))

    def abort(self, partition_id: int):
        self._check(self._lib.vpca_pool_abort(self._h, int(partition_id)))

    def reduceAndFinalize(self):
        self._check(self._lib.vpca_pool_reduce_and_finalize(self._h))

    def getGram(self) -> np.ndarray:
        out = np.empty((self.n, self.n), dtype=np.int32)
        self._check(self._lib.vpca_pool_get_gram(self._h, _host_ptr(out)))
        return out

    def computePca(self, k: int = 2):
        flat = np.empty(self.n * k, dtype=np.float64)
        evals = np.empty(k, dtype=np.float64)
        nz = ctypes.c_int32(0)
        self._check(self._lib.vpca_pool_compute_pca(self._h, int(k), _host_ptr(flat), _host_ptr(evals), ctypes.byref(nz)))
        return flat.reshape(k, self.n).T.copy(), evals, int(nz.value)

    def stats(self) -> dict:
        st = VpcaStats()
        self._check(self._lib.vpca_pool_get_stats(self._h, ctypes.byref(st)))
        return {name: getattr(st, name) for name, _ in VpcaStats._fields_}
