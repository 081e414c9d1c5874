"""
ctypes binding of libh2b200.so -- the C ABI declared in include/h2b200.h.

The product library is CUDA-only (sm_100a).  There is no CPU fallback: if the shared library is
missing, or no Blackwell GPU is usable, loading / initialisation raises.  The CPU "kernel-logic
emulator" build (tools/emu, used by unit tests of the kernel sources) is refused here unless a test
asks for it explicitly with `allow_emulator=True`.
"""
from __future__ import annotations

import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
DEFAULT_LIB = os.path.join(_HERE, "lib", "libh2b200.so")

H2B_OK = 0


class H2BError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("h2b200 error %d: %s" % (code, msg))
        self.code = code


_EXPORTS = [
    "h2b_init", "h2b_init_device", "h2b_shutdown", "h2b_device_count", "h2b_last_error", "h2b_version",
    "h2b_is_emulator", "h2b_msm_bn254_g1", "h2b_ntt_bn254_fr", "h2b_register_bases", "h2b_unregister_bases",
    "h2b_msm_bn254_g1_registered", "h2b_ntt_bn254_fr_dev", "h2b_msm_bn254_g1_dev",
    "h2b_msm_bn254_g1_dev_partial", "h2b_msm_fold_partials", "h2b_msm_fold_partials_dev", "h2b_fr_scale_dev",
    "h2b_dev_alloc", "h2b_dev_free", "h2b_memcpy_h2d", "h2b_memcpy_d2h", "h2b_memcpy_h2d_async", "h2b_dev_sync", "h2b_gen_points_dev",
    "h2b_gen_scalars_dev", "h2b_field_op", "h2b_ec_op", "h2b_imad_bench", "h2b_set_msm_window",
    "h2b_launch_count", "h2b_profile_enable", "h2b_profile_read", "h2b_msm_bn254_g1_dev_registered",
    "h2b_set_msm_precomp", "h2b_base_set_info", "h2b_msm_bn254_g1_batch_registered", "h2b_ntt_bn254_fr_batch",
    "h2b_lagrange_to_coeff_dev", "h2b_coeff_to_extended_dev", "h2b_extended_to_coeff_dev",
    "h2b_fr_batch_invert_dev", "h2b_fr_prefix_product_dev", "h2b_fr_eval_polynomial_dev", "h2b_fr_kate_division_dev",
    "h2b_fr_lincomb_dev", "h2b_fr_transpose_dev", "h2b_permutation_product_dev", "h2b_lookup_product_dev", "h2b_lookup_permute_dev", "h2b_lookup_permute_async_dev", "h2b_g1_decode_dev", "h2b_g1_encode_dev", "h2b_srs_read", "h2b_srs_write", "h2b_srs_cache_clear",
    "h2b_evaluate_graph_dev", "h2b_evaluate_graph_shard_dev", "h2b_evaluate_h_permutation_shard_dev", "h2b_evaluate_h_lookup_shard_dev", "h2b_evaluate_h_permutation_dev", "h2b_evaluate_h_lookup_dev", "h2b_evaluate_graph_info",
    "h2b_register_bases_sharded", "h2b_msm_bn254_g1_dev_batch_registered", "h2b_implicit_cache_stats", "h2b_msm_checksum_dev", "h2b_ntt_bn254_fr_dev_batch", "h2b_lagrange_to_coeff_dev_batch", "h2b_coeff_to_extended_dev_batch", "h2b_memcpy_d2d_async", "h2b_memset_zero_async", "h2b_column_pipeline",
    "h2b_srs_setup", "h2b_g1_generator_mul_dev", "h2b_g1_to_lagrange_dev", "h2b_srs_downsize",
    "h2b_permutation_sigma_dev", "h2b_keygen_lagrange_indicators_dev", "h2b_permutation_build_vk", "h2b_permutation_build_pk",
    "h2b_selector_exclusion", "h2b_keygen_fixed_build_vk", "h2b_keygen_fixed_build_pk",
    "h2b_pk_create", "h2b_keygen_fixed_build_pk_resident", "h2b_permutation_build_pk_resident", "h2b_keygen_lagrange_indicators_resident",
    "h2b_pk_put_lagrange", "h2b_pk_column", "h2b_pk_download", "h2b_pk_info", "h2b_pk_release",
    "h2b_fr_eval_queries_dev", "h2b_shplonk_begin", "h2b_shplonk_finish", "h2b_shplonk_release",
]

# include/h2b200.h enums of the resident proving key
PK_FIXED, PK_PERMUTATION, PK_INDICATORS = 0, 1, 2
PK_VALUES, PK_COEFF, PK_EXTENDED = 0, 1, 2
PK_REPLICATED, PK_ROW_SHARDED = 0, 1


# ---- include/h2b200.h structs of the quotient evaluation ------------------------------------------------
class ValueSourceStruct(ctypes.Structure):
    _fields_ = [("kind", ctypes.c_uint32), ("index", ctypes.c_uint32), ("rotation", ctypes.c_uint32)]


class CalculationStruct(ctypes.Structure):
    _fields_ = [("op", ctypes.c_uint32), ("target", ctypes.c_uint32), ("a", ValueSourceStruct), ("b", ValueSourceStruct),
                ("parts_offset", ctypes.c_uint32), ("parts_len", ctypes.c_uint32)]


class GraphStruct(ctypes.Structure):
    _fields_ = [("constants", ctypes.c_void_p), ("n_constants", ctypes.c_uint32),
                ("rotations", ctypes.c_void_p), ("n_rotations", ctypes.c_uint32),
                ("calculations", ctypes.c_void_p), ("n_calculations", ctypes.c_uint32),
                ("parts", ctypes.c_void_p), ("n_parts", ctypes.c_uint32),
                ("n_intermediates", ctypes.c_uint32)]


class EvalColumnsStruct(ctypes.Structure):
    _fields_ = [("fixed", ctypes.c_void_p), ("n_fixed", ctypes.c_uint32),
                ("advice", ctypes.c_void_p), ("n_advice", ctypes.c_uint32),
                ("instance", ctypes.c_void_p), ("n_instance", ctypes.c_uint32),
                ("challenges", ctypes.c_void_p), ("n_challenges", ctypes.c_uint32),
                ("beta", ctypes.c_void_p), ("gamma", ctypes.c_void_p), ("theta", ctypes.c_void_p), ("y", ctypes.c_void_p)]


class OpeningQueryStruct(ctypes.Structure):
    _fields_ = [("poly", ctypes.c_uint32), ("reserved", ctypes.c_uint32), ("point", ctypes.c_uint64 * 4)]


def _queries(queries):
    """[(poly index, point words)] -> a ctypes array of h2b_opening_query"""
    arr = (OpeningQueryStruct * max(len(queries), 1))()
    for i, (poly, point) in enumerate(queries):
        arr[i].poly = int(poly)
        arr[i].point[:] = [int(w) for w in np.asarray(point, dtype=np.uint64).reshape(4)]
    return arr


class ShardStruct(ctypes.Structure):
    _fields_ = [("row0", ctypes.c_uint32), ("rows", ctypes.c_uint32), ("halo", ctypes.c_uint32)]


assert ctypes.sizeof(CalculationStruct) == 40


class GraphArrays:
    """A GraphEvaluator flattened into the arrays h2b_graph points at (kept alive by this object)."""

    def __init__(self, constants, rotations, calculations, parts, n_intermediates: int):
        self.constants = np.ascontiguousarray(constants, dtype=np.uint64).reshape(-1, 4)
        self.rotations = np.ascontiguousarray(rotations, dtype=np.int32).reshape(-1)
        self.calculations = np.ascontiguousarray(calculations, dtype=np.uint32).reshape(-1, 10)
        self.parts = np.ascontiguousarray(parts, dtype=np.uint32).reshape(-1, 3)
        self.n_intermediates = int(n_intermediates)

    def struct(self) -> GraphStruct:
        return GraphStruct(self.constants.ctypes.data, self.constants.shape[0], self.rotations.ctypes.data, self.rotations.shape[0],
                           self.calculations.ctypes.data, self.calculations.shape[0], self.parts.ctypes.data, self.parts.shape[0],
                           self.n_intermediates)


class EvalColumns:
    """Device pointers of the fixed / advice / instance cosets plus the scalars of one evaluate_h call."""

    def __init__(self, fixed, advice, instance, challenges, beta, gamma, theta, y):
        self.fixed = np.array(list(fixed), dtype=np.uint64)
        self.advice = np.array(list(advice), dtype=np.uint64)
        self.instance = np.array(list(instance), dtype=np.uint64)
        self.challenges = np.ascontiguousarray(challenges, dtype=np.uint64).reshape(-1, 4)
        self.beta, self.gamma, self.theta, self.y = (np.ascontiguousarray(v, dtype=np.uint64).reshape(4) for v in (beta, gamma, theta, y))

    def struct(self) -> EvalColumnsStruct:
        return EvalColumnsStruct(self.fixed.ctypes.data, self.fixed.shape[0], self.advice.ctypes.data, self.advice.shape[0],
                                 self.instance.ctypes.data, self.instance.shape[0], self.challenges.ctypes.data, self.challenges.shape[0],
                                 self.beta.ctypes.data, self.gamma.ctypes.data, self.theta.ctypes.data, self.y.ctypes.data)


def exported_symbols():
    """Every symbol include/h2b200.h declares (checked by the CPU test-suite against the built .so)."""
    return list(_EXPORTS)


def _u64(a: np.ndarray) -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=np.uint64)
    return a


def _ptr_array(ptrs):
    return (ctypes.c_void_p * len(ptrs))(*ptrs)


def _mapping_columns(mapping, k: int):
    """a permutation mapping -- (P, 2^k, 2) uint64 or a list of (2^k, 2) columns of (column, row) pairs -> contiguous columns"""
    cols = [_u64(c).reshape(-1, 2) for c in mapping]
    for c in cols:
        assert c.shape[0] == 1 << k, "mapping column of %d rows, expected 2^%d" % (c.shape[0], k)
    return cols


def _activation_rows(activations, k: int):
    """selector activations -- (S, 2^k) bool / uint8 or a list of such rows -> contiguous uint8 rows (Rust's Vec<bool> layout)"""
    rows = [np.ascontiguousarray(np.asarray(a).reshape(-1), dtype=np.uint8) for a in activations]
    for r in rows:
        assert r.shape[0] == 1 << k, "activation row of %d entries, expected 2^%d" % (r.shape[0], k)
    return rows


def _fixed_args(fixed, activations, combination_of, root_of, k: int):
    fx = [_u64(c).reshape(-1, 4) for c in fixed]
    for c in fx:
        assert c.shape[0] == 1 << k, "fixed column of %d rows, expected 2^%d" % (c.shape[0], k)
    acts = _activation_rows(activations, k)
    co = np.ascontiguousarray(np.asarray(combination_of, dtype=np.uint32).reshape(-1))
    ro = np.ascontiguousarray(np.asarray(root_of, dtype=np.uint32).reshape(-1))
    assert co.shape[0] == len(acts) and ro.shape[0] == len(acts), "one combination and one root per selector"
    return fx, acts, co, ro


class Lib:
    def __init__(self, path: str | None = None, allow_emulator: bool = False):
        path = path or os.environ.get("H2B200_LIB", DEFAULT_LIB)
        if not os.path.exists(path):
            raise FileNotFoundError(
                "libh2b200.so not found at %s -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). There is no CPU fallback." % path)
        self.path = path
        L = ctypes.CDLL(path)
        vp, sz, u64, u32, i32 = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int
        L.h2b_init.argtypes = [i32]
        L.h2b_init_device.argtypes = [i32]
        L.h2b_shutdown.restype = None
        L.h2b_last_error.restype = ctypes.c_char_p
        L.h2b_version.restype = ctypes.c_char_p
        L.h2b_msm_bn254_g1.argtypes = [vp, vp, sz, vp]
        L.h2b_ntt_bn254_fr.argtypes = [vp, vp, u32]
        L.h2b_register_bases.argtypes = [vp, sz, ctypes.POINTER(u64)]
        L.h2b_unregister_bases.argtypes = [u64]
        L.h2b_register_bases_sharded.argtypes = [vp, sz, ctypes.POINTER(u64)]
        L.h2b_msm_bn254_g1_dev_batch_registered.argtypes = [i32, vp, vp, sz, u64, vp, vp]
        L.h2b_implicit_cache_stats.argtypes = [vp]
        L.h2b_msm_checksum_dev.argtypes = [i32, vp, u64, u64, sz, vp, vp]
        L.h2b_msm_bn254_g1_registered.argtypes = [vp, u64, sz, sz, vp]
        L.h2b_ntt_bn254_fr_dev.argtypes = [i32, vp, vp, u32, vp]
        L.h2b_ntt_bn254_fr_dev_batch.argtypes = [i32, vp, sz, vp, u32, vp]
        L.h2b_msm_bn254_g1_dev.argtypes = [i32, vp, vp, sz, vp, vp]
        L.h2b_msm_bn254_g1_dev_partial.argtypes = [i32, vp, vp, sz, vp, vp]
        L.h2b_msm_bn254_g1_dev_registered.argtypes = [i32, vp, u64, sz, sz, vp, vp]
        L.h2b_set_msm_precomp.argtypes = [i32]
        L.h2b_base_set_info.argtypes = [u64, ctypes.POINTER(u32), ctypes.POINTER(u32), ctypes.POINTER(u64)]
        L.h2b_msm_bn254_g1_batch_registered.argtypes = [vp, vp, sz, u64, vp]
        L.h2b_ntt_bn254_fr_batch.argtypes = [vp, sz, vp, u32]
        L.h2b_msm_fold_partials.argtypes = [i32, vp, sz, vp]
        L.h2b_msm_fold_partials_dev.argtypes = [i32, vp, sz, vp, vp]
        L.h2b_fr_scale_dev.argtypes = [i32, vp, sz, vp, i32, vp]
        L.h2b_fr_batch_invert_dev.argtypes = [i32, vp, sz, vp]
        L.h2b_fr_prefix_product_dev.argtypes = [i32, vp, vp, sz, vp]
        L.h2b_fr_eval_polynomial_dev.argtypes = [i32, vp, sz, vp, vp, vp]
        L.h2b_fr_kate_division_dev.argtypes = [i32, vp, sz, vp, vp, vp]
        L.h2b_lagrange_to_coeff_dev.argtypes = [i32, vp, u32, vp, vp, vp]
        L.h2b_coeff_to_extended_dev.argtypes = [i32, vp, u32, u32, vp, vp, vp]
        L.h2b_extended_to_coeff_dev.argtypes = [i32, vp, u32, vp, vp, vp]
        L.h2b_lagrange_to_coeff_dev_batch.argtypes = [i32, vp, sz, u32, vp, vp, vp]
        L.h2b_coeff_to_extended_dev_batch.argtypes = [i32, vp, sz, u32, u32, vp, vp, vp]
        L.h2b_fr_lincomb_dev.argtypes = [i32, vp, vp, u32, sz, vp, vp]
        L.h2b_fr_transpose_dev.argtypes = [i32, vp, vp, u32, u32, vp]
        L.h2b_permutation_product_dev.argtypes = [i32, vp, vp, u32, sz, vp, vp, vp, vp, vp, vp, vp, vp]
        L.h2b_lookup_product_dev.argtypes = [i32, vp, vp, vp, vp, sz, vp, vp, vp, vp]
        L.h2b_lookup_permute_dev.argtypes = [i32, vp, vp, u32, vp, vp, vp]
        L.h2b_lookup_permute_async_dev.argtypes = [i32, vp, vp, u32, vp, vp, vp, vp]
        L.h2b_g1_decode_dev.argtypes = [i32, vp, sz, i32, vp, ctypes.POINTER(u64), vp]
        L.h2b_g1_encode_dev.argtypes = [i32, vp, sz, vp, vp]
        L.h2b_srs_read.argtypes = [ctypes.c_char_p, i32, ctypes.POINTER(u32), vp, vp, vp, sz, ctypes.POINTER(sz), ctypes.POINTER(u64), ctypes.POINTER(u64)]
        L.h2b_srs_write.argtypes = [ctypes.c_char_p, i32, u32, vp, vp, vp, sz]
        L.h2b_srs_setup.argtypes = [u32, vp, vp, vp, ctypes.POINTER(u64), ctypes.POINTER(u64)]
        L.h2b_g1_generator_mul_dev.argtypes = [i32, vp, sz, vp, vp]
        L.h2b_g1_to_lagrange_dev.argtypes = [i32, vp, u32, vp, vp]
        L.h2b_srs_downsize.argtypes = [u64, u32, vp, ctypes.POINTER(u64), ctypes.POINTER(u64)]
        L.h2b_permutation_sigma_dev.argtypes = [i32, vp, u32, u32, vp, vp, vp, vp, vp]
        L.h2b_keygen_lagrange_indicators_dev.argtypes = [i32, u32, u32, u32, vp, vp, vp, vp, vp, vp, vp, vp]
        L.h2b_permutation_build_vk.argtypes = [vp, u32, u32, vp, vp, u64, vp]
        L.h2b_permutation_build_pk.argtypes = [vp, u32, u32, u32, vp, vp, vp, vp, vp, vp, vp, vp, vp]
        L.h2b_selector_exclusion.argtypes = [vp, u32, u32, vp]
        L.h2b_keygen_fixed_build_vk.argtypes = [vp, u32, vp, u32, vp, vp, u32, u32, u64, vp]
        L.h2b_keygen_fixed_build_pk.argtypes = [vp, u32, vp, u32, vp, vp, u32, u32, u32, vp, vp, vp, vp, vp, vp, vp]
        L.h2b_pk_create.argtypes = [u32, u32, u32, u32, i32, u32, vp, vp, vp, vp, vp, ctypes.POINTER(u64)]
        L.h2b_keygen_fixed_build_pk_resident.argtypes = [vp, u32, vp, u32, vp, vp, u32, u64, u32]
        L.h2b_permutation_build_pk_resident.argtypes = [vp, u32, vp, u64]
        L.h2b_keygen_lagrange_indicators_resident.argtypes = [u64, u32]
        L.h2b_pk_put_lagrange.argtypes = [u64, i32, u32, u32, vp]
        L.h2b_pk_column.argtypes = [u64, i32, i32, i32, u32, ctypes.POINTER(vp), vp]
        L.h2b_pk_download.argtypes = [u64, i32, i32, u32, vp]
        L.h2b_pk_info.argtypes = [u64, vp]
        L.h2b_pk_release.argtypes = [u64]
        L.h2b_fr_eval_queries_dev.argtypes = [i32, vp, u32, sz, vp, u32, vp, vp]
        L.h2b_shplonk_begin.argtypes = [i32, vp, i32, u32, sz, vp, u32, u64, vp, vp, vp, ctypes.POINTER(u64)]
        L.h2b_shplonk_finish.argtypes = [u64, vp, vp]
        L.h2b_shplonk_release.argtypes = [u64]
        L.h2b_evaluate_graph_dev.argtypes = [i32, vp, vp, vp, u32, i32, vp]
        L.h2b_evaluate_h_permutation_dev.argtypes = [i32, vp, u32, i32, vp, u32, vp, vp, u32, u32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
        L.h2b_evaluate_h_lookup_dev.argtypes = [i32, vp, vp, vp, u32, i32, vp, vp, vp, vp, vp, vp, vp]
        L.h2b_evaluate_graph_shard_dev.argtypes = [i32, vp, vp, vp, u32, i32, vp, vp]
        L.h2b_evaluate_h_permutation_shard_dev.argtypes = [i32, vp, u32, i32, vp, u32, vp, vp, u32, u32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
        L.h2b_evaluate_h_lookup_shard_dev.argtypes = [i32, vp, vp, vp, u32, i32, vp, vp, vp, vp, vp, vp, vp, vp]
        L.h2b_evaluate_graph_info.argtypes = [ctypes.POINTER(u32), ctypes.POINTER(u32)]
        L.h2b_dev_alloc.argtypes = [i32, sz, ctypes.POINTER(vp)]
        L.h2b_dev_free.argtypes = [i32, vp]
        L.h2b_memcpy_h2d.argtypes = [i32, vp, vp, sz]
        L.h2b_memcpy_d2h.argtypes = [i32, vp, vp, sz]
        L.h2b_memcpy_h2d_async.argtypes = [i32, vp, vp, sz, vp]
        L.h2b_memcpy_d2d_async.argtypes = [i32, vp, vp, sz, vp]
        L.h2b_memset_zero_async.argtypes = [i32, vp, sz, vp]
        L.h2b_column_pipeline.argtypes = [i32, vp, u64, u32, u32, vp, vp, vp, vp, vp, vp, vp, ctypes.POINTER(vp)]
        L.h2b_dev_sync.argtypes = [i32]
        L.h2b_gen_points_dev.argtypes = [i32, u64, sz, vp, vp]
        L.h2b_gen_scalars_dev.argtypes = [i32, u64, sz, i32, vp, vp]
        L.h2b_field_op.argtypes = [i32, i32, vp, vp, sz, vp]
        L.h2b_ec_op.argtypes = [i32, vp, vp, sz, vp]
        L.h2b_imad_bench.argtypes = [i32, i32, i32, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_double)]
        L.h2b_set_msm_window.argtypes = [i32]
        L.h2b_launch_count.restype = ctypes.c_ulonglong
        L.h2b_profile_enable.argtypes = [i32, i32]
        L.h2b_profile_read.argtypes = [i32, vp, vp, i32, ctypes.POINTER(i32)]
        self.L = L
        self.is_emulator = bool(L.h2b_is_emulator())
        if self.is_emulator and not allow_emulator:
            raise RuntimeError("%s is the CPU kernel-logic emulator build; the product path only runs the CUDA library" % path)

    # ---- helpers ------------------------------------------------------------------------------
    def check(self, rc: int):
        if rc != H2B_OK:
            raise H2BError(rc, (self.L.h2b_last_error() or b"").decode())

    def version(self) -> str:
        return self.L.h2b_version().decode()

    # ---- lifecycle ------------------------------------------------------------------------------
    def init(self, n_devices: int = 0):
        self.check(self.L.h2b_init(n_devices))

    def init_device(self, device: int):
        self.check(self.L.h2b_init_device(device))

    def shutdown(self):
        self.L.h2b_shutdown()

    def device_count(self) -> int:
        return self.L.h2b_device_count()

    # ---- host-pointer drop-ins ------------------------------------------------------------------
    def msm(self, scalars: np.ndarray, bases: np.ndarray) -> np.ndarray:
        scalars, bases = _u64(scalars), _u64(bases)
        n = scalars.shape[0] if scalars.ndim > 1 else scalars.size // 4
        nb = bases.shape[0] if bases.ndim > 1 else bases.size // 8
        if n != nb:
            raise AssertionError("best_multiexp: coeffs.len() != bases.len() (%d vs %d)" % (n, nb))
        out = np.zeros(12, dtype=np.uint64)
        self.check(self.L.h2b_msm_bn254_g1(scalars.ctypes.data, bases.ctypes.data, n, out.ctypes.data))
        return out

    def ntt(self, a: np.ndarray, omega: np.ndarray, log_n: int) -> np.ndarray:
        """In place on a C-contiguous uint64 (2^log_n, 4) array; returns it."""
        assert a.dtype == np.uint64 and a.flags["C_CONTIGUOUS"]
        assert a.size == 4 << log_n, "best_fft: a.len() != 1 << log_n"
        omega = _u64(omega)
        self.check(self.L.h2b_ntt_bn254_fr(a.ctypes.data, omega.ctypes.data, log_n))
        return a

    def register_bases(self, bases: np.ndarray) -> int:
        bases = _u64(bases)
        h = ctypes.c_uint64(0)
        self.check(self.L.h2b_register_bases(bases.ctypes.data, bases.size // 8, ctypes.byref(h)))
        return h.value

    def register_bases_sharded(self, bases: np.ndarray) -> int:
        """Rows split over the devices (device d keeps [d n/D, (d+1) n/D) and its tables): the point-range mode."""
        bases = _u64(bases)
        h = ctypes.c_uint64(0)
        self.check(self.L.h2b_register_bases_sharded(bases.ctypes.data, bases.size // 8, ctypes.byref(h)))
        return h.value

    def implicit_cache_stats(self) -> dict:
        out = np.zeros(6, dtype=np.uint64)
        self.check(self.L.h2b_implicit_cache_stats(out.ctypes.data))
        return dict(zip(("uploads", "hits", "stale", "direct", "sets", "sets_with_tables"), (int(v) for v in out)))

    def unregister_bases(self, handle: int):
        self.check(self.L.h2b_unregister_bases(handle))

    def msm_registered(self, scalars: np.ndarray, handle: int, offset: int = 0) -> np.ndarray:
        scalars = _u64(scalars)
        out = np.zeros(12, dtype=np.uint64)
        self.check(self.L.h2b_msm_bn254_g1_registered(scalars.ctypes.data, handle, offset, scalars.size // 4, out.ctypes.data))
        return out

    def msm_batch_registered(self, columns, handle: int) -> np.ndarray:
        """columns: list of (n_j, 4) uint64 arrays -> (len(columns), 12) Jacobian results"""
        cols = [_u64(c).reshape(-1, 4) for c in columns]
        ptrs = (ctypes.c_void_p * len(cols))(*[c.ctypes.data for c in cols])
        lens = (ctypes.c_size_t * len(cols))(*[c.shape[0] for c in cols])
        out = np.zeros((len(cols), 12), dtype=np.uint64)
        self.check(self.L.h2b_msm_bn254_g1_batch_registered(ptrs, lens, len(cols), handle, out.ctypes.data))
        return out

    def ntt_batch(self, polys, omega: np.ndarray, log_n: int):
        """In place on each C-contiguous uint64 (2^log_n, 4) array of the list."""
        for a in polys:
            assert a.dtype == np.uint64 and a.flags["C_CONTIGUOUS"] and a.size == 4 << log_n
        ptrs = (ctypes.c_void_p * len(polys))(*[a.ctypes.data for a in polys])
        omega = _u64(omega)
        self.check(self.L.h2b_ntt_bn254_fr_batch(ptrs, len(polys), omega.ctypes.data, log_n))
        return polys

    # ---- device-pointer entry points ------------------------------------------------------------
    def ntt_dev(self, device: int, d_a: int, omega: np.ndarray, log_n: int, stream: int = 0):
        omega = _u64(omega)
        self.check(self.L.h2b_ntt_bn254_fr_dev(device, d_a, omega.ctypes.data, log_n, stream))

    def ntt_dev_batch(self, device: int, d_polys, omega: np.ndarray, log_n: int, stream: int = 0):
        """d_polys: device pointers of equally sized polynomials, transformed in place by shared pass launches"""
        omega = _u64(omega)
        ptrs = (ctypes.c_void_p * len(d_polys))(*d_polys)
        self.check(self.L.h2b_ntt_bn254_fr_dev_batch(device, ptrs, len(d_polys), omega.ctypes.data, log_n, stream))

    def msm_dev(self, device: int, d_scalars: int, d_bases: int, n: int, d_out: int, stream: int = 0):
        self.check(self.L.h2b_msm_bn254_g1_dev(device, d_scalars, d_bases, n, d_out, stream))

    def msm_dev_partial(self, device: int, d_scalars: int, d_bases: int, n: int, d_out_block: int, stream: int = 0):
        self.check(self.L.h2b_msm_bn254_g1_dev_partial(device, d_scalars, d_bases, n, d_out_block, stream))

    def msm_dev_registered(self, device: int, d_scalars: int, handle: int, offset: int, n: int, d_out_block: int, stream: int = 0):
        self.check(self.L.h2b_msm_bn254_g1_dev_registered(device, d_scalars, handle, offset, n, d_out_block, stream))

    def msm_dev_batch_registered(self, device: int, d_columns, lens, handle: int, d_out_blocks: int, stream: int = 0):
        """d_columns: device pointers, lens: scalars per column; d_out_blocks: len(d_columns) x 224 bytes on the device"""
        ptrs = (ctypes.c_void_p * len(d_columns))(*d_columns)
        ln = (ctypes.c_size_t * len(d_columns))(*lens)
        self.check(self.L.h2b_msm_bn254_g1_dev_batch_registered(device, ptrs, ln, len(d_columns), handle, d_out_blocks, stream))

    def msm_checksum_dev(self, device: int, d_scalars: int, seed: int, n: int, d_out: int, first: int = 0, stream: int = 0):
        """sum_i s_i z_i mod r (canonical, 32 B at d_out) for the synthetic points P_i = [z_i]G of gen_points(seed)"""
        self.check(self.L.h2b_msm_checksum_dev(device, d_scalars, seed, first, n, d_out, stream))

    def set_msm_precomp(self, spacing: int):
        self.check(self.L.h2b_set_msm_precomp(spacing))

    def base_set_info(self, handle: int):
        nt, sp, by = ctypes.c_uint32(0), ctypes.c_uint32(0), ctypes.c_uint64(0)
        self.check(self.L.h2b_base_set_info(handle, ctypes.byref(nt), ctypes.byref(sp), ctypes.byref(by)))
        return {"n_tables": nt.value, "spacing": sp.value, "device_bytes": by.value}

    def msm_fold_partials(self, blocks: np.ndarray, device: int = 0) -> np.ndarray:
        blocks = _u64(blocks).reshape(-1, 28)
        out = np.zeros(12, dtype=np.uint64)
        self.check(self.L.h2b_msm_fold_partials(device, blocks.ctypes.data, blocks.shape[0], out.ctypes.data))
        return out

    def msm_fold_partials_dev(self, device: int, d_blocks: int, count: int, d_out: int, stream: int = 0):
        self.check(self.L.h2b_msm_fold_partials_dev(device, d_blocks, count, d_out, stream))

    def fr_scale_dev(self, device: int, d_a: int, n: int, factors: np.ndarray, stream: int = 0):
        factors = _u64(factors).reshape(-1, 4)
        self.check(self.L.h2b_fr_scale_dev(device, d_a, n, factors.ctypes.data, factors.shape[0], stream))

    def lagrange_to_coeff_dev(self, device: int, d_a: int, k: int, omega_inv: np.ndarray, ifft_divisor: np.ndarray, stream: int = 0):
        omega_inv, ifft_divisor = _u64(omega_inv), _u64(ifft_divisor)
        self.check(self.L.h2b_lagrange_to_coeff_dev(device, d_a, k, omega_inv.ctypes.data, ifft_divisor.ctypes.data, stream))

    def coeff_to_extended_dev(self, device: int, d_a: int, k: int, extended_k: int, extended_omega: np.ndarray, zeta_powers: np.ndarray, stream: int = 0):
        extended_omega, zeta_powers = _u64(extended_omega), _u64(zeta_powers).reshape(3, 4)
        self.check(self.L.h2b_coeff_to_extended_dev(device, d_a, k, extended_k, extended_omega.ctypes.data, zeta_powers.ctypes.data, stream))

    def lagrange_to_coeff_dev_batch(self, device: int, d_cols, k: int, omega_inv: np.ndarray, ifft_divisor: np.ndarray, stream: int = 0):
        omega_inv, ifft_divisor = _u64(omega_inv), _u64(ifft_divisor)
        ptrs = (ctypes.c_void_p * len(d_cols))(*d_cols)
        self.check(self.L.h2b_lagrange_to_coeff_dev_batch(device, ptrs, len(d_cols), k, omega_inv.ctypes.data, ifft_divisor.ctypes.data, stream))

    def coeff_to_extended_dev_batch(self, device: int, d_cols, k: int, extended_k: int, extended_omega: np.ndarray, zeta_powers: np.ndarray, stream: int = 0):
        extended_omega, zeta_powers = _u64(extended_omega), _u64(zeta_powers).reshape(3, 4)
        ptrs = (ctypes.c_void_p * len(d_cols))(*d_cols)
        self.check(self.L.h2b_coeff_to_extended_dev_batch(device, ptrs, len(d_cols), k, extended_k, extended_omega.ctypes.data, zeta_powers.ctypes.data, stream))

    def column_pipeline(self, lagrange: np.ndarray, handle_g_lagrange: int, k: int, extended_k: int, omega_inv, ifft_divisor, extended_omega, zeta_powers,
                        want_coeff: bool = True, want_extended: bool = True, keep_on_device: bool = False, device: int = 0):
        """commit_lagrange + lagrange_to_coeff + coeff_to_extended of one host column with a single upload
        -> dict(commitment (12 words), coeff, extended, d_extended)"""
        lagrange = _u64(lagrange).reshape(-1, 4)
        assert lagrange.shape[0] == 1 << k
        w = [_u64(v) for v in (omega_inv, ifft_divisor, extended_omega)]
        zp = _u64(zeta_powers).reshape(3, 4)
        out = np.zeros(12, dtype=np.uint64)
        coeff = np.empty((1 << k, 4), dtype=np.uint64) if want_coeff else None
        ext = np.empty((1 << extended_k, 4), dtype=np.uint64) if want_extended else None
        d_ext = ctypes.c_void_p(0)
        self.check(self.L.h2b_column_pipeline(device, lagrange.ctypes.data, handle_g_lagrange, k, extended_k, w[0].ctypes.data, w[1].ctypes.data,
                                              w[2].ctypes.data, zp.ctypes.data, out.ctypes.data, coeff.ctypes.data if want_coeff else None,
                                              ext.ctypes.data if want_extended else None, ctypes.byref(d_ext) if keep_on_device else None))
        return dict(commitment=out, coeff=coeff, extended=ext, d_extended=d_ext.value)

    def extended_to_coeff_dev(self, device: int, d_a: int, extended_k: int, extended_omega_inv: np.ndarray, factors: np.ndarray, stream: int = 0):
        extended_omega_inv, factors = _u64(extended_omega_inv), _u64(factors).reshape(3, 4)
        self.check(self.L.h2b_extended_to_coeff_dev(device, d_a, extended_k, extended_omega_inv.ctypes.data, factors.ctypes.data, stream))

    def fr_batch_invert_dev(self, device: int, d_a: int, n: int, stream: int = 0):
        self.check(self.L.h2b_fr_batch_invert_dev(device, d_a, n, stream))

    def fr_prefix_product_dev(self, device: int, d_in: int, d_out: int, n: int, stream: int = 0):
        self.check(self.L.h2b_fr_prefix_product_dev(device, d_in, d_out, n, stream))

    def _column_op(self, a: np.ndarray, op, device: int = 0) -> np.ndarray:
        a = _u64(a).reshape(-1, 4)
        n = a.shape[0]
        out = np.empty_like(a)
        d = self.dev_alloc(device, max(n, 1) * 32)
        try:
            if n:
                self.h2d(device, d, a)
                op(d, n)
                self.dev_sync(device)
                self.d2h(device, out, d)
        finally:
            self.dev_free(device, d)
        return out

    def fr_batch_invert(self, a: np.ndarray, device: int = 0) -> np.ndarray:
        """a[i] -> 1 / a[i] (zeros stay zero), through device memory"""
        return self._column_op(a, lambda d, n: self.fr_batch_invert_dev(device, d, n), device)

    def fr_prefix_product(self, a: np.ndarray, device: int = 0) -> np.ndarray:
        """out[0] = 1, out[i] = a[0] * ... * a[i-1], through device memory (in place on the device)"""
        return self._column_op(a, lambda d, n: self.fr_prefix_product_dev(device, d, d, n), device)

    def fr_eval_polynomial(self, coeffs: np.ndarray, x: np.ndarray, device: int = 0) -> np.ndarray:
        """eval_polynomial(poly, point) through device memory -> (4,) uint64"""
        coeffs, x = _u64(coeffs).reshape(-1, 4), _u64(x)
        n = coeffs.shape[0]
        out = np.zeros(4, dtype=np.uint64)
        d, d_o = self.dev_alloc(device, max(n, 1) * 32), self.dev_alloc(device, 32)
        try:
            if n:
                self.h2d(device, d, coeffs)
            self.check(self.L.h2b_fr_eval_polynomial_dev(device, d, n, x.ctypes.data, d_o, 0))
            self.dev_sync(device)
            self.d2h(device, out, d_o)
        finally:
            self.dev_free(device, d)
            self.dev_free(device, d_o)
        return out

    def fr_kate_division(self, a: np.ndarray, b: np.ndarray, device: int = 0) -> np.ndarray:
        """kate_division(a, b) through device memory -> (n - 1, 4) uint64"""
        a, b = _u64(a).reshape(-1, 4), _u64(b)
        n = a.shape[0]
        q = np.zeros((max(n - 1, 0), 4), dtype=np.uint64)
        if n <= 1:
            return q
        d, d_q = self.dev_alloc(device, n * 32), self.dev_alloc(device, n * 32)
        try:
            self.h2d(device, d, a)
            self.check(self.L.h2b_fr_kate_division_dev(device, d, n, b.ctypes.data, d_q, 0))
            self.dev_sync(device)
            self.d2h(device, q, d_q)
        finally:
            self.dev_free(device, d)
            self.dev_free(device, d_q)
        return q

    # ---- grand products (permutation / lookup z polynomials) -------------------------------------------
    def permutation_product_dev(self, device: int, d_values, d_permutations, n: int, beta, gamma, delta, deltaomega, omega, last_z, d_z: int,
                                stream: int = 0):
        v, p = np.array(list(d_values), dtype=np.uint64), np.array(list(d_permutations), dtype=np.uint64)
        assert v.shape == p.shape
        w = [np.ascontiguousarray(x, dtype=np.uint64).reshape(4) for x in (beta, gamma, delta, deltaomega, omega, last_z)]
        self.check(self.L.h2b_permutation_product_dev(device, v.ctypes.data, p.ctypes.data, v.shape[0], n, *[x.ctypes.data for x in w], d_z, stream))

    def lookup_product_dev(self, device: int, d_compressed_input: int, d_compressed_table: int, d_permuted_input: int, d_permuted_table: int, n: int,
                           beta, gamma, d_z: int, stream: int = 0):
        w = [np.ascontiguousarray(x, dtype=np.uint64).reshape(4) for x in (beta, gamma)]
        self.check(self.L.h2b_lookup_product_dev(device, d_compressed_input, d_compressed_table, d_permuted_input, d_permuted_table, n,
                                                 w[0].ctypes.data, w[1].ctypes.data, d_z, stream))

    def fr_lincomb_dev(self, device: int, d_cols, coeffs, n: int, d_out: int, stream: int = 0):
        p = np.array(list(d_cols), dtype=np.uint64)
        c = _u64(coeffs).reshape(-1, 4)
        assert c.shape[0] == p.shape[0]
        self.check(self.L.h2b_fr_lincomb_dev(device, p.ctypes.data if p.size else None, c.ctypes.data if c.size else None, p.shape[0], n, d_out, stream))

    def fr_transpose(self, a: np.ndarray, device: int = 0) -> np.ndarray:
        """(rows, cols, 4) uint64 matrix of Fr elements -> its transpose (cols, rows, 4), through the device"""
        a = np.ascontiguousarray(a, dtype=np.uint64)
        rows, cols = a.shape[0], a.shape[1]
        out = np.empty((cols, rows, 4), dtype=np.uint64)
        if rows == 0 or cols == 0:
            return out
        d_in, d_out = self.dev_alloc(device, a.nbytes), self.dev_alloc(device, a.nbytes)
        try:
            self.h2d(device, d_in, a)
            self.check(self.L.h2b_fr_transpose_dev(device, d_in, d_out, rows, cols, None))
            self.dev_sync(device)
            self.d2h(device, out, d_out)
        finally:
            self.dev_free(device, d_in)
            self.dev_free(device, d_out)
        return out

    def fr_lincomb(self, cols, coeffs, device: int = 0) -> np.ndarray:
        """sum_j coeffs[j] * cols[j], host arrays in and out"""
        n = _u64(cols[0]).size // 4
        return self._columns_op(list(cols), n, lambda d, d_out: self.fr_lincomb_dev(device, d, coeffs, n, d_out), device)

    def lookup_permute_dev(self, device: int, d_input: int, d_table: int, usable_rows: int, d_permuted_input: int, d_permuted_table: int, stream: int = 0):
        self.check(self.L.h2b_lookup_permute_dev(device, d_input, d_table, usable_rows, d_permuted_input, d_permuted_table, stream))

    def lookup_permute_async_dev(self, device: int, d_input: int, d_table: int, usable_rows: int, d_permuted_input: int, d_permuted_table: int,
                                 d_status: int, stream: int = 0):
        self.check(self.L.h2b_lookup_permute_async_dev(device, d_input, d_table, usable_rows, d_permuted_input, d_permuted_table, d_status, stream))

    def lookup_permute(self, input_expression, table_expression, usable_rows: int, device: int = 0):
        """permute_expression_pair on host arrays -> (permuted_input, permuted_table), usable_rows x 4 each"""
        a, t = _u64(input_expression).reshape(-1, 4), _u64(table_expression).reshape(-1, 4)
        n = a.shape[0]
        assert t.shape[0] == n and usable_rows <= n
        d = [self.dev_alloc(device, max(n, 1) * 32) for _ in range(4)]
        try:
            self.h2d(device, d[0], a)
            self.h2d(device, d[1], t)
            self.lookup_permute_dev(device, d[0], d[1], usable_rows, d[2], d[3])
            pa, pt = np.empty((usable_rows, 4), dtype=np.uint64), np.empty((usable_rows, 4), dtype=np.uint64)
            if usable_rows:
                self.d2h(device, pa, d[2])
                self.d2h(device, pt, d[3])
            return pa, pt
        finally:
            for p in d:
                self.dev_free(device, p)

    def _columns_op(self, cols, n: int, op, device: int = 0) -> np.ndarray:
        """upload `cols` (n x 4 each), run op(device pointers, d_out), download n x 4"""
        held = []
        try:
            for c in cols:
                d = self.dev_alloc(device, max(n, 1) * 32)
                held.append(d)
                if n:
                    self.h2d(device, d, _u64(c).reshape(-1, 4))
            d_out = self.dev_alloc(device, max(n, 1) * 32)
            held.append(d_out)
            op(held[:-1], d_out)
            self.dev_sync(device)
            out = np.empty((n, 4), dtype=np.uint64)
            if n:
                self.d2h(device, out, d_out)
            return out
        finally:
            for d in held:
                self.dev_free(device, d)

    def permutation_product(self, values, permutations, beta, gamma, delta, deltaomega, omega, last_z, device: int = 0) -> np.ndarray:
        """permutation::Argument::commit for one set, host arrays in and out (z without the blinding rows)"""
        m, n = len(values), _u64(values[0]).size // 4
        return self._columns_op(list(values) + list(permutations), n,
                                lambda d, d_z: self.permutation_product_dev(device, d[:m], d[m:], n, beta, gamma, delta, deltaomega, omega, last_z, d_z),
                                device)

    def lookup_product(self, compressed_input, compressed_table, permuted_input, permuted_table, beta, gamma, device: int = 0) -> np.ndarray:
        n = _u64(compressed_input).size // 4
        return self._columns_op([compressed_input, compressed_table, permuted_input, permuted_table], n,
                                lambda d, d_z: self.lookup_product_dev(device, d[0], d[1], d[2], d[3], n, beta, gamma, d_z), device)

    # ---- SRS on-disk format ---------------------------------------------------------------------------
    def g1_decode(self, data: np.ndarray, fmt: int, device: int = 0) -> np.ndarray:
        """encoded points ((n, 32) uint8 compressed or (n, 64) raw) -> (n, 8) uint64 affine; raises H2BError on an invalid point"""
        data = np.ascontiguousarray(data, dtype=np.uint8)
        ps = 32 if fmt == 0 else 64
        n = data.size // ps
        out = np.empty((n, 8), dtype=np.uint64)
        d_in, d_out = self.dev_alloc(device, max(n, 1) * ps), self.dev_alloc(device, max(n, 1) * 64)
        try:
            if n:
                self.h2d(device, d_in, data)
            bad = ctypes.c_uint64(0)
            self.check(self.L.h2b_g1_decode_dev(device, d_in, n, fmt, d_out, ctypes.byref(bad), 0))
            if n:
                self.d2h(device, out, d_out)
        finally:
            self.dev_free(device, d_in)
            self.dev_free(device, d_out)
        return out

    def g1_encode(self, aff: np.ndarray, device: int = 0) -> np.ndarray:
        """(n, 8) uint64 affine -> (n, 32) uint8 compressed (G1Affine::to_bytes)"""
        aff = _u64(aff).reshape(-1, 8)
        n = aff.shape[0]
        out = np.empty((n, 32), dtype=np.uint8)
        d_in, d_out = self.dev_alloc(device, max(n, 1) * 64), self.dev_alloc(device, max(n, 1) * 32)
        try:
            if n:
                self.h2d(device, d_in, aff)
                self.check(self.L.h2b_g1_encode_dev(device, d_in, n, d_out, 0))
                self.dev_sync(device)
                self.d2h(device, out, d_out)
        finally:
            self.dev_free(device, d_in)
            self.dev_free(device, d_out)
        return out

    def srs_read(self, path: str, fmt: int, want_host: bool = True, register: bool = True):
        """-> dict(k, g, g_lagrange, g2_bytes, handle_g, handle_g_lagrange); see h2b_srs_read"""
        with open(path, "rb") as f:
            k0 = int.from_bytes(f.read(4), "little")
        # the header is untrusted: size the host arrays only after the file length agrees with it (the library checks again)
        point = 32 if fmt == 0 else 64
        if k0 > 28 or os.path.getsize(path) < 4 + 2 * (1 << k0) * point + 4 * point:
            raise H2BError(-2, "h2b_srs_read: %s is shorter than its header (k = %d) promises" % (path, k0))
        n = 1 << k0
        g = np.empty((n, 8), dtype=np.uint64) if want_host else None
        gl = np.empty((n, 8), dtype=np.uint64) if want_host else None
        g2 = np.zeros(256, dtype=np.uint8)
        k, g2_len, hg, hl = ctypes.c_uint32(0), ctypes.c_size_t(0), ctypes.c_uint64(0), ctypes.c_uint64(0)
        self.check(self.L.h2b_srs_read(path.encode(), fmt, ctypes.byref(k), g.ctypes.data if want_host else None, gl.ctypes.data if want_host else None,
                                       g2.ctypes.data, g2.size, ctypes.byref(g2_len), ctypes.byref(hg) if register else None,
                                       ctypes.byref(hl) if register else None))
        return dict(k=k.value, g=g, g_lagrange=gl, g2_bytes=bytes(g2[:g2_len.value]), handle_g=hg.value, handle_g_lagrange=hl.value)

    def srs_cache_clear(self):
        self.check(self.L.h2b_srs_cache_clear())

    def srs_write(self, path: str, fmt: int, k: int, g: np.ndarray, g_lagrange: np.ndarray, g2_bytes: bytes):
        g, g_lagrange = _u64(g).reshape(-1, 8), _u64(g_lagrange).reshape(-1, 8)
        assert g.shape[0] == 1 << k and g_lagrange.shape[0] == 1 << k
        buf = np.frombuffer(g2_bytes, dtype=np.uint8).copy()
        self.check(self.L.h2b_srs_write(path.encode(), fmt, k, g.ctypes.data, g_lagrange.ctypes.data, buf.ctypes.data if buf.size else None, buf.size))

    def srs_setup(self, k: int, s, want_host: bool = True, register: bool = True):
        """ParamsKZG::setup with toxic waste s (4 words, Montgomery) -> the dict of srs_read (g2_bytes empty: G2 is the caller's)"""
        s = _u64(s).reshape(4)
        n = 1 << k if 0 <= k <= 28 else 0
        g = np.empty((n, 8), dtype=np.uint64) if want_host else None
        gl = np.empty((n, 8), dtype=np.uint64) if want_host else None
        hg, hl = ctypes.c_uint64(0), ctypes.c_uint64(0)
        self.check(self.L.h2b_srs_setup(k, s.ctypes.data, g.ctypes.data if want_host else None, gl.ctypes.data if want_host else None,
                                        ctypes.byref(hg) if register else None, ctypes.byref(hl) if register else None))
        return dict(k=k, g=g, g_lagrange=gl, g2_bytes=b"", handle_g=hg.value, handle_g_lagrange=hl.value)

    def g1_generator_mul_dev(self, device: int, d_scalars: int, n: int, d_out: int, stream: int = 0):
        self.check(self.L.h2b_g1_generator_mul_dev(device, d_scalars, n, d_out, stream))

    def g1_generator_mul(self, scalars: np.ndarray, device: int = 0) -> np.ndarray:
        """(n, 4) Montgomery scalars -> (n, 8) affine [scalar] G, through device memory"""
        scalars = _u64(scalars).reshape(-1, 4)
        n = scalars.shape[0]
        out = np.empty((n, 8), dtype=np.uint64)
        d_s, d_o = self.dev_alloc(device, max(n, 1) * 32), self.dev_alloc(device, max(n, 1) * 64)
        try:
            if n:
                self.h2d(device, d_s, scalars)
                self.g1_generator_mul_dev(device, d_s, n, d_o)
                self.dev_sync(device)
                self.d2h(device, out, d_o)
        finally:
            self.dev_free(device, d_s)
            self.dev_free(device, d_o)
        return out

    def g1_to_lagrange_dev(self, device: int, d_g: int, k: int, d_out: int, stream: int = 0):
        self.check(self.L.h2b_g1_to_lagrange_dev(device, d_g, k, d_out, stream))

    def g1_to_lagrange(self, points: np.ndarray, k: int, device: int = 0) -> np.ndarray:
        """g_to_lagrange of the first 2^k of the (n, 8) affine points -> (2^k, 8) affine, through device memory"""
        points = _u64(points).reshape(-1, 8)
        n = 1 << k
        assert points.shape[0] >= n
        out = np.empty((n, 8), dtype=np.uint64)
        d_p = self.dev_alloc(device, n * 64)
        try:
            self.h2d(device, d_p, points[:n])
            self.g1_to_lagrange_dev(device, d_p, k, d_p)
            self.dev_sync(device)
            self.d2h(device, out, d_p)
        finally:
            self.dev_free(device, d_p)
        return out

    def srs_downsize(self, handle_g: int, k: int, want_host: bool = True, register: bool = True):
        """ParamsKZG::downsize of the resident g of a replicated set -> dict(g_lagrange (host copy or None), handle_g,
        handle_g_lagrange) with new sets for the 2^k-point prefix of g and its g_lagrange (0 when not registered)"""
        gl = np.empty((1 << k, 8), dtype=np.uint64) if want_host and 0 <= k <= 28 else None
        hg, hl = ctypes.c_uint64(0), ctypes.c_uint64(0)
        self.check(self.L.h2b_srs_downsize(handle_g, k, gl.ctypes.data if gl is not None else None,
                                           ctypes.byref(hg) if register else None, ctypes.byref(hl) if register else None))
        return dict(g_lagrange=gl, handle_g=hg.value, handle_g_lagrange=hl.value)

    # ---- key generation: permutation sigma columns and keygen_pk's indicator columns -------------------------------
    def permutation_sigma_dev(self, device: int, d_mapping, k: int, delta, omega, d_sigma, d_status: int, stream: int = 0):
        """sigma of len(d_mapping) mapping columns (device pointers, n x 16 B each) into d_sigma; the status word at d_status is
        1 + the flat index of an out-of-range entry, 0 when all are valid (read it after synchronising `stream`)"""
        m, s = _ptr_array(d_mapping), _ptr_array(d_sigma)
        w = [_u64(x).reshape(4) for x in (delta, omega)]
        self.check(self.L.h2b_permutation_sigma_dev(device, m, len(d_mapping), k, w[0].ctypes.data, w[1].ctypes.data, s, d_status, stream))

    def keygen_lagrange_indicators_dev(self, device: int, k: int, extended_k: int, blinding_factors: int, omega_inv, ifft_divisor, extended_omega,
                                       zeta_powers, d_l0: int, d_l_last: int, d_l_active_row: int, stream: int = 0):
        w = [_u64(x).reshape(4) for x in (omega_inv, ifft_divisor, extended_omega)]
        zp = _u64(zeta_powers).reshape(3, 4)
        self.check(self.L.h2b_keygen_lagrange_indicators_dev(device, k, extended_k, blinding_factors, w[0].ctypes.data, w[1].ctypes.data, w[2].ctypes.data,
                                                             zp.ctypes.data, d_l0, d_l_last, d_l_active_row, stream))

    def keygen_lagrange_indicators(self, k: int, extended_k: int, blinding_factors: int, omega_inv, ifft_divisor, extended_omega, zeta_powers,
                                   device: int = 0):
        """(l0, l_last, l_active_row) of keygen_pk, each (2^extended_k, 4), computed on the device and downloaded"""
        en = 1 << extended_k
        outs = [np.empty((en, 4), dtype=np.uint64) for _ in range(3)]
        d = [self.dev_alloc(device, en * 32) for _ in range(3)]
        try:
            self.keygen_lagrange_indicators_dev(device, k, extended_k, blinding_factors, omega_inv, ifft_divisor, extended_omega, zeta_powers, *d)
            self.dev_sync(device)
            for o, p in zip(outs, d):
                self.d2h(device, o, p)
        finally:
            for p in d:
                self.dev_free(device, p)
        return tuple(outs)

    def permutation_build_vk(self, mapping, k: int, delta, omega, handle_g_lagrange: int) -> np.ndarray:
        """Assembly::build_vk: mapping (P, 2^k, 2) uint64 (or a list of (2^k, 2) columns) -> (P, 12) Jacobian commitments"""
        cols = _mapping_columns(mapping, k)
        w = [_u64(x).reshape(4) for x in (delta, omega)]
        out = np.zeros((len(cols), 12), dtype=np.uint64)
        self.check(self.L.h2b_permutation_build_vk(_ptr_array([c.ctypes.data for c in cols]), len(cols), k, w[0].ctypes.data, w[1].ctypes.data,
                                                   handle_g_lagrange, out.ctypes.data))
        return out

    def permutation_build_pk(self, mapping, k: int, extended_k: int, delta, omega, omega_inv, ifft_divisor, extended_omega, zeta_powers,
                             want_permutations: bool = True, want_polys: bool = True, want_cosets: bool = True):
        """Assembly::build_pk -> dict(permutations, polys, cosets): lists of (2^k, 4), (2^k, 4) and (2^extended_k, 4) arrays (None when not wanted)"""
        cols = _mapping_columns(mapping, k)
        P, n = len(cols), 1 << k
        w = [_u64(x).reshape(4) for x in (delta, omega, omega_inv, ifft_divisor, extended_omega)]
        zp = _u64(zeta_powers).reshape(3, 4)
        perms = [np.empty((n, 4), dtype=np.uint64) for _ in range(P)] if want_permutations else None
        polys = [np.empty((n, 4), dtype=np.uint64) for _ in range(P)] if want_polys else None
        cosets = [np.empty((1 << extended_k, 4), dtype=np.uint64) for _ in range(P)] if want_cosets else None
        arr = lambda xs: _ptr_array([x.ctypes.data for x in xs]) if xs is not None else None
        self.check(self.L.h2b_permutation_build_pk(_ptr_array([c.ctypes.data for c in cols]), P, k, extended_k, *[x.ctypes.data for x in w],
                                                   zp.ctypes.data, arr(perms), arr(polys), arr(cosets)))
        return dict(permutations=perms, polys=polys, cosets=cosets)

    # ---- key generation: compress_selectors' exclusion matrix and the fixed columns of keygen_vk / keygen_pk ---------------------
    def selector_exclusion(self, activations, k: int) -> np.ndarray:
        """process's exclusion matrix: activations (S, 2^k) bool / uint8 (or a list of such rows) -> (S, S) bool, True where two
        selectors are active on a common row (symmetric, False on the diagonal)"""
        acts = _activation_rows(activations, k)
        out = np.zeros((len(acts), len(acts)), dtype=np.uint8)
        self.check(self.L.h2b_selector_exclusion(_ptr_array([a.ctypes.data for a in acts]) if acts else None, len(acts), k, out.ctypes.data))
        return out.astype(bool)

    def keygen_fixed_build_vk(self, fixed, activations, combination_of, root_of, n_combinations: int, k: int, handle_g_lagrange: int) -> np.ndarray:
        """keygen_vk's fixed commitments: fixed (F, 2^k, 4) Montgomery words (or a list of (2^k, 4) columns), activations (S, 2^k) and
        the assignment -> (F + n_combinations, 12) Jacobian commitments of the fixed columns, then the combination columns"""
        fx, acts, co, ro = _fixed_args(fixed, activations, combination_of, root_of, k)
        out = np.zeros((len(fx) + n_combinations, 12), dtype=np.uint64)
        self.check(self.L.h2b_keygen_fixed_build_vk(_ptr_array([c.ctypes.data for c in fx]) if fx else None, len(fx),
                                                    _ptr_array([a.ctypes.data for a in acts]) if acts else None, len(acts), co.ctypes.data,
                                                    ro.ctypes.data, n_combinations, k, handle_g_lagrange, out.ctypes.data))
        return out

    def keygen_fixed_build_pk(self, fixed, activations, combination_of, root_of, n_combinations: int, k: int, extended_k: int, omega_inv, ifft_divisor,
                              extended_omega, zeta_powers, want_values: bool = True, want_polys: bool = True, want_cosets: bool = True):
        """keygen_pk's fixed columns -> dict(combination_values, polys, cosets): the n_combinations combination columns (2^k, 4), and
        lagrange_to_coeff / coeff_to_extended of all F + n_combinations columns ((2^k, 4) and (2^extended_k, 4)); None when not wanted"""
        fx, acts, co, ro = _fixed_args(fixed, activations, combination_of, root_of, k)
        n, T = 1 << k, len(fx) + n_combinations
        w = [_u64(x).reshape(4) for x in (omega_inv, ifft_divisor, extended_omega)]
        zp = _u64(zeta_powers).reshape(3, 4)
        vals = [np.empty((n, 4), dtype=np.uint64) for _ in range(n_combinations)] if want_values else None
        polys = [np.empty((n, 4), dtype=np.uint64) for _ in range(T)] if want_polys else None
        cosets = [np.empty((1 << extended_k, 4), dtype=np.uint64) for _ in range(T)] if want_cosets else None
        arr = lambda xs: _ptr_array([x.ctypes.data for x in xs]) if xs else None
        self.check(self.L.h2b_keygen_fixed_build_pk(arr(fx), len(fx), arr(acts), len(acts), co.ctypes.data, ro.ctypes.data, n_combinations, k, extended_k,
                                                    *[x.ctypes.data for x in w], zp.ctypes.data, arr(vals), arr(polys), arr(cosets)))
        return dict(combination_values=vals, polys=polys, cosets=cosets)

    # ---- the proving key resident on the devices ---------------------------------------------------------------------------------
    def pk_create(self, k: int, extended_k: int, n_fixed: int, n_permutation: int, layout: int, halo: int, omega, omega_inv, ifft_divisor,
                  extended_omega, zeta_powers) -> int:
        w = [_u64(x).reshape(4) for x in (omega, omega_inv, ifft_divisor, extended_omega)]
        zp = _u64(zeta_powers).reshape(3, 4)
        h = ctypes.c_uint64(0)
        self.check(self.L.h2b_pk_create(k, extended_k, n_fixed, n_permutation, layout, halo, *[x.ctypes.data for x in w], zp.ctypes.data, ctypes.byref(h)))
        return h.value

    def keygen_fixed_build_pk_resident(self, fixed, activations, combination_of, root_of, n_combinations: int, k: int, pk: int, first_column: int = 0):
        fx, acts, co, ro = _fixed_args(fixed, activations, combination_of, root_of, k)
        arr = lambda xs: _ptr_array([x.ctypes.data for x in xs]) if xs else None
        self.check(self.L.h2b_keygen_fixed_build_pk_resident(arr(fx), len(fx), arr(acts), len(acts), co.ctypes.data, ro.ctypes.data, n_combinations, pk,
                                                             first_column))

    def permutation_build_pk_resident(self, mapping, k: int, delta, pk: int):
        cols = _mapping_columns(mapping, k)
        dl = _u64(delta).reshape(4)
        self.check(self.L.h2b_permutation_build_pk_resident(_ptr_array([c.ctypes.data for c in cols]), len(cols), dl.ctypes.data, pk))

    def keygen_lagrange_indicators_resident(self, pk: int, blinding_factors: int):
        self.check(self.L.h2b_keygen_lagrange_indicators_resident(pk, blinding_factors))

    def pk_put_lagrange(self, pk: int, part: int, first: int, values, k: int):
        cols = [_u64(c).reshape(-1, 4) for c in values]
        for c in cols:
            assert c.shape[0] == 1 << k, "column of %d rows, expected 2^%d" % (c.shape[0], k)
        self.check(self.L.h2b_pk_put_lagrange(pk, part, first, len(cols), _ptr_array([c.ctypes.data for c in cols]) if cols else None))

    def pk_column(self, pk: int, device: int, part: int, form: int, index: int):
        """-> (device pointer, (row0, rows, halo)) of one column on `device`"""
        p, sh = ctypes.c_void_p(0), ShardStruct()
        self.check(self.L.h2b_pk_column(pk, device, part, form, index, ctypes.byref(p), ctypes.addressof(sh)))
        return p.value or 0, (sh.row0, sh.rows, sh.halo)

    def pk_download(self, pk: int, part: int, form: int, index: int, rows: int) -> np.ndarray:
        out = np.empty((rows, 4), dtype=np.uint64)
        self.check(self.L.h2b_pk_download(pk, part, form, index, out.ctypes.data))
        return out

    def pk_info(self, pk: int) -> list:
        """-> bytes the pk holds on each device"""
        out = np.zeros(max(self.device_count(), 1), dtype=np.uint64)
        self.check(self.L.h2b_pk_info(pk, out.ctypes.data))
        return [int(x) for x in out]

    def pk_release(self, pk: int):
        self.check(self.L.h2b_pk_release(pk))

    # ---- the multi-point opening (SHPLONK) ---------------------------------------------------------------
    def eval_queries_dev(self, device: int, d_polys, n: int, queries, d_out: int, stream: int = 0):
        """eval_polynomial of every query (poly index into d_polys, point words) -> d_out, one Fr per query"""
        ptrs = _ptr_array(list(d_polys))
        q = _queries(queries)
        self.check(self.L.h2b_fr_eval_queries_dev(device, ptrs, len(d_polys), n, q, len(queries), d_out, stream))

    def shplonk_begin(self, device: int, polys, on_host: bool, n: int, queries, handle_g: int, y, v):
        """polys: host arrays (on_host) or device pointers -> (h1 Jacobian, session handle)"""
        ptrs = _ptr_array([p.ctypes.data for p in polys] if on_host else list(polys))
        q = _queries(queries)
        y, v = _u64(y).reshape(4), _u64(v).reshape(4)
        out = np.zeros(12, dtype=np.uint64)
        h = ctypes.c_uint64(0)
        self.check(self.L.h2b_shplonk_begin(device, ptrs, 1 if on_host else 0, len(polys), n, q, len(queries), handle_g, y.ctypes.data, v.ctypes.data,
                                            out.ctypes.data, ctypes.byref(h)))
        return out, h.value

    def shplonk_finish(self, session: int, u) -> np.ndarray:
        u = _u64(u).reshape(4)
        out = np.zeros(12, dtype=np.uint64)
        self.check(self.L.h2b_shplonk_finish(session, u.ctypes.data, out.ctypes.data))
        return out

    def shplonk_release(self, session: int):
        self.check(self.L.h2b_shplonk_release(session))

    # ---- quotient evaluation (evaluate_h) on device-resident extended-coset columns ------------------
    def evaluate_graph_dev(self, device: int, graph: GraphArrays, cols: EvalColumns, d_values: int, size: int, rot_scale: int, stream: int = 0,
                           shard=None):
        """shard = (row0, rows, halo): the row-sharded variant (column pointers are slices with halo, d_values the halo-free slice)"""
        g, c = graph.struct(), cols.struct()
        if shard is None:
            self.check(self.L.h2b_evaluate_graph_dev(device, ctypes.addressof(g), ctypes.addressof(c), d_values, size, rot_scale, stream))
        else:
            sh = ShardStruct(*shard)
            self.check(self.L.h2b_evaluate_graph_shard_dev(device, ctypes.addressof(g), ctypes.addressof(c), d_values, size, rot_scale,
                                                           ctypes.addressof(sh), stream))

    def evaluate_h_permutation_dev(self, device: int, d_values: int, size: int, rot_scale: int, product_cosets, columns, perm_cosets, chunk_len: int,
                                   last_rotation: int, d_l0: int, d_l_last: int, d_l_active_row: int, beta, gamma, y, delta, zeta, extended_omega,
                                   stream: int = 0, shard=None):
        pc, co, pe = (np.array(list(v), dtype=np.uint64) for v in (product_cosets, columns, perm_cosets))
        assert co.shape[0] == pe.shape[0]
        w = [np.ascontiguousarray(v, dtype=np.uint64).reshape(4) for v in (beta, gamma, y, delta, zeta, extended_omega)]
        args = [device, d_values, size, rot_scale, pc.ctypes.data, pc.shape[0], co.ctypes.data, pe.ctypes.data, co.shape[0], chunk_len, last_rotation, d_l0,
                d_l_last, d_l_active_row, *[v.ctypes.data for v in w]]
        if shard is None:
            self.check(self.L.h2b_evaluate_h_permutation_dev(*args, stream))
        else:
            sh = ShardStruct(*shard)
            self.check(self.L.h2b_evaluate_h_permutation_shard_dev(*args, ctypes.addressof(sh), stream))

    def evaluate_h_lookup_dev(self, device: int, graph: GraphArrays, cols: EvalColumns, d_values: int, size: int, rot_scale: int, d_product: int,
                              d_permuted_input: int, d_permuted_table: int, d_l0: int, d_l_last: int, d_l_active_row: int, stream: int = 0, shard=None):
        g, c = graph.struct(), cols.struct()
        args = [device, ctypes.addressof(g), ctypes.addressof(c), d_values, size, rot_scale, d_product, d_permuted_input, d_permuted_table, d_l0, d_l_last,
                d_l_active_row]
        if shard is None:
            self.check(self.L.h2b_evaluate_h_lookup_dev(*args, stream))
        else:
            sh = ShardStruct(*shard)
            self.check(self.L.h2b_evaluate_h_lookup_shard_dev(*args, ctypes.addressof(sh), stream))

    def evaluate_graph_info(self):
        """-> (live-value slots, micro-operations) of the graph this thread compiled last"""
        a, b = ctypes.c_uint32(0), ctypes.c_uint32(0)
        self.check(self.L.h2b_evaluate_graph_info(ctypes.byref(a), ctypes.byref(b)))
        return a.value, b.value

    def dev_alloc(self, device: int, nbytes: int) -> int:
        p = ctypes.c_void_p(0)
        self.check(self.L.h2b_dev_alloc(device, nbytes, ctypes.byref(p)))
        return p.value or 0

    def dev_free(self, device: int, p: int):
        self.check(self.L.h2b_dev_free(device, p))

    def h2d(self, device: int, d_dst: int, src: np.ndarray):
        src = np.ascontiguousarray(src)
        self.check(self.L.h2b_memcpy_h2d(device, d_dst, src.ctypes.data, src.nbytes))

    def h2d_async(self, device: int, d_dst: int, src: np.ndarray, stream: int = 0):
        """upload into a buffer nothing in flight touches, without draining the device first; `src` must be contiguous"""
        assert src.flags["C_CONTIGUOUS"]
        self.check(self.L.h2b_memcpy_h2d_async(device, d_dst, src.ctypes.data, src.nbytes, stream))

    def d2h(self, device: int, dst: np.ndarray, d_src: int):
        assert dst.flags["C_CONTIGUOUS"]
        self.check(self.L.h2b_memcpy_d2h(device, dst.ctypes.data, d_src, dst.nbytes))

    def dev_sync(self, device: int = 0):
        self.check(self.L.h2b_dev_sync(device))

    # ---- synthetic workload + diagnostics -----------------------------------------------------------
    def gen_points_dev(self, device: int, seed: int, n: int, d_out: int, stream: int = 0):
        self.check(self.L.h2b_gen_points_dev(device, seed, n, d_out, stream))

    def gen_scalars_dev(self, device: int, seed: int, n: int, kind: int, d_out: int, stream: int = 0):
        self.check(self.L.h2b_gen_scalars_dev(device, seed, n, kind, d_out, stream))

    def gen_points(self, seed: int, n: int, device: int = 0) -> np.ndarray:
        out = np.empty((n, 8), dtype=np.uint64)
        d = self.dev_alloc(device, max(n, 1) * 64)
        try:
            self.gen_points_dev(device, seed, n, d)
            self.dev_sync(device)
            if n:
                self.d2h(device, out, d)
        finally:
            self.dev_free(device, d)
        return out

    def gen_scalars(self, seed: int, n: int, kind: int = 0, device: int = 0) -> np.ndarray:
        out = np.empty((n, 4), dtype=np.uint64)
        d = self.dev_alloc(device, max(n, 1) * 32)
        try:
            self.gen_scalars_dev(device, seed, n, kind, d)
            self.dev_sync(device)
            if n:
                self.d2h(device, out, d)
        finally:
            self.dev_free(device, d)
        return out

    def field_op(self, field: str, op: str, a: np.ndarray, b: np.ndarray | None = None) -> np.ndarray:
        a = _u64(a)
        b = a if b is None else _u64(b)
        out = np.empty_like(a)
        ops = {"add": 0, "sub": 1, "mul": 2, "sqr": 3, "inv": 4, "from_mont": 5, "to_mont": 6,
               "mul_lazy": 7, "sqr_lazy": 8, "add_lazy": 9, "sub_lazy": 10, "canon": 11, "is_zero_lazy": 12}
        self.check(self.L.h2b_field_op({"fr": 0, "fq": 1}[field], ops[op], a.ctypes.data, b.ctypes.data, a.size // 4, out.ctypes.data))
        return out

    def ec_op(self, op: int, p: np.ndarray, q: np.ndarray) -> np.ndarray:
        p, q = _u64(p), _u64(q)
        out = np.empty_like(p)
        self.check(self.L.h2b_ec_op(op, p.ctypes.data, q.ctypes.data, p.size // 8, out.ctypes.data))
        return out

    def imad_bench(self, kind: int, iters: int, device: int = 0):
        ms, ops = ctypes.c_float(0), ctypes.c_double(0)
        self.check(self.L.h2b_imad_bench(device, kind, iters, ctypes.byref(ms), ctypes.byref(ops)))
        return ms.value, ops.value

    def launch_count(self) -> int:
        return int(self.L.h2b_launch_count())

    def profile_enable(self, on: bool, device: int = 0):
        self.check(self.L.h2b_profile_enable(device, 1 if on else 0))

    def profile_read(self, device: int = 0):
        """-> list of (tag, ms) in launch order; clears the record."""
        cap = 8192
        tags = np.zeros(cap, dtype=np.int32)
        ms = np.zeros(cap, dtype=np.float32)
        cnt = ctypes.c_int(0)
        self.check(self.L.h2b_profile_read(device, tags.ctypes.data, ms.ctypes.data, cap, ctypes.byref(cnt)))
        return [(int(tags[i]), float(ms[i])) for i in range(cnt.value)]

    def set_msm_window(self, c: int):
        self.check(self.L.h2b_set_msm_window(c))


_default: Lib | None = None


def load(path: str | None = None, allow_emulator: bool = False) -> Lib:
    """Load (once) and return the product library. Raises if it is missing -- there is no fallback."""
    global _default
    if path is not None or allow_emulator:
        return Lib(path, allow_emulator)
    if _default is None:
        _default = Lib()
    return _default
