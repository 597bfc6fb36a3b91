"""halo2_vectordb_b200 -- B200 (sm_100a) backend for the KZG-commit / EvaluationDomain hot path of
erhant/halo2-vectordb's keygen / prove flow (/root/reference/src/scaffold/mod.rs:273,296).

This module is the Python host-side mirror of the upstream interface the C ABI (include/h2v.h)
stands in for -- halo2-axiom `arithmetic::{best_multiexp, best_fft}`, `poly::kzg::commitment::ParamsKZG`
and `poly::domain::EvaluationDomain` -- with the same names, argument meaning and error behaviour
(upstream `assert!` panics become `ValueError`).  It is a thin ctypes layer: all arithmetic runs in
libh2v.so's CUDA kernels.  There is no CPU fallback and nothing here imports `oracle/`; if the
native library is missing, importing the compute API raises.

Data convention = halo2curves: numpy uint64 arrays of little-endian limbs in Montgomery form,
Fr (n, 4), G1Affine (n, 8), G1 Jacobian (12,).
"""
import ctypes as C
import os
from collections import namedtuple

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libh2v.so")

H2V_BASIS_MONOMIAL, H2V_BASIS_LAGRANGE = 0, 1
OP_LAGRANGE_TO_COEFF, OP_COEFF_TO_LAGRANGE, OP_COEFF_TO_EXTENDED, OP_EXTENDED_TO_COEFF, OP_DIVIDE_BY_VANISHING = range(5)
KERNEL_CLASSES = ["msm_digits", "msm_scan", "msm_scatter", "msm_accumulate", "msm_finish", "msm_reduce", "msm_final", "ntt"]

# every symbol include/h2v.h declares (tests check the library exports all of them)
ABI_SYMBOLS = [
    "h2v_init", "h2v_device_list", "h2v_dev_alloc_on", "h2v_device_count", "h2v_last_error", "h2v_version", "h2v_host_register", "h2v_host_unregister", "h2v_dev_alloc", "h2v_dev_free", "h2v_dev_upload", "h2v_dev_download",
    "h2v_srs_load", "h2v_srs_setup", "h2v_srs_free", "h2v_srs_info", "h2v_commit", "h2v_commit_batch", "h2v_commit_batch_dev", "h2v_best_multiexp", "h2v_g1_sum",
    "h2v_best_fft", "h2v_domain_new", "h2v_domain_free", "h2v_domain_k", "h2v_domain_extended_k", "h2v_domain_constant",
    "h2v_lagrange_to_coeff", "h2v_coeff_to_lagrange", "h2v_coeff_to_extended", "h2v_extended_to_coeff",
    "h2v_divide_by_vanishing_poly", "h2v_domain_transform_batch", "h2v_domain_transform_dev",
    "h2v_eval_polynomial_batch", "h2v_eval_polynomial_dev", "h2v_batch_invert", "h2v_grand_product", "h2v_grand_product_dev", "h2v_kate_division",
    "h2v_permute_expression_pair", "h2v_permute_expression_pair_dev", "h2v_permute_expression_pair_batch_dev",
    "h2v_quotient_gates_dev", "h2v_quotient_permutation_dev", "h2v_quotient_lookup_dev",
    "h2v_g1_to_bytes", "h2v_fr_to_repr",
    "h2v_domain_rotate_omega", "h2v_domain_rotate_extended", "h2v_domain_l_i_range", "h2v_domain_fill", "h2v_kate_division_dev",
    "h2v_quotient_gates_ptrs_dev", "h2v_quotient_permutation_ptrs_dev", "h2v_quotient_permutation_range_ptrs_dev", "h2v_commit_batch_resident",
    "h2v_pk_load", "h2v_pk_free", "h2v_create_proof", "h2v_create_proofs", "h2v_proof_size", "h2v_pk_last_phase_ms",
    "h2v_mock_prover", "h2v_pk_mock_prover", "h2v_mock_last_ms",
    "h2v_witness_program_new", "h2v_witness_program_free", "h2v_witness_program_info", "h2v_witness_program_inputs",
    "h2v_witness_program_rule_counts",
    "h2v_witness_generate", "h2v_witness_last_ms", "h2v_create_proofs_from_inputs", "h2v_pk_mock_prover_from_inputs",
    "h2v_transcript_new", "h2v_transcript_free", "h2v_transcript_common_point", "h2v_transcript_common_scalar",
    "h2v_transcript_write_point", "h2v_transcript_write_scalar", "h2v_transcript_squeeze_challenge", "h2v_transcript_bytes",
    "h2v_poseidon_permutation", "h2v_poseidon_permutation_variant", "h2v_chacha20_fr_random", "h2v_chacha20_block",
    "h2v_srs_gen", "h2v_g2_mul_generator", "h2v_srs_write_file", "h2v_srs_read_file",
    "h2v_selftest_field", "h2v_selftest_group", "h2v_synthetic_bases", "h2v_selftest_imad_peak", "h2v_selftest_imad_probe", "h2v_selftest_op_rate", "h2v_set_tuning", "h2v_launch_count", "h2v_last_kernel_ms", "h2v_last_msm_entries",
]
BUILDER_SYMBOLS = [      # the circuit builder (halo2_vectordb_b200.circuit)
    "h2v_builder_new", "h2v_builder_free", "h2v_builder_quantize", "h2v_builder_dequantize", "h2v_builder_assign_witnesses",
    "h2v_builder_load_constant", "h2v_builder_cell_values", "h2v_builder_make_public", "h2v_builder_call",
    "h2v_builder_nearest_vector", "h2v_builder_kmeans", "h2v_builder_poseidon_new", "h2v_builder_poseidon_hash",
    "h2v_builder_merkle_commitment", "h2v_builder_stats", "h2v_builder_config", "h2v_builder_trace", "h2v_builder_layout",
    "h2v_layout_free", "h2v_layout_info", "h2v_layout_columns", "h2v_layout_instance", "h2v_layout_break_points",
    "h2v_builder_new_recording",
]
ABI_SYMBOLS += BUILDER_SYMBOLS


class H2VError(RuntimeError):
    pass


_lib = None
_u64p = C.POINTER(C.c_uint64)


def lib():
    """Load libh2v.so (built in-tree by halo2_vectordb_b200.build / __graft_entry__.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise H2VError(f"{LIB_PATH} is missing: run `python -m halo2_vectordb_b200.build` "
                           "(there is no CPU fallback for this path)")
        L = C.CDLL(LIB_PATH)
        L.h2v_last_error.restype = C.c_char_p
        L.h2v_version.restype = C.c_char_p
        L.h2v_launch_count.restype = C.c_uint64
        L.h2v_domain_k.restype = C.c_uint32
        L.h2v_domain_extended_k.restype = C.c_uint32
        L.h2v_domain_k.argtypes = [C.c_void_p]
        L.h2v_domain_extended_k.argtypes = [C.c_void_p]
        L.h2v_init.argtypes = [C.POINTER(C.c_int), C.c_int]
        L.h2v_device_list.argtypes = [C.POINTER(C.c_int), C.c_int]
        L.h2v_dev_alloc_on.argtypes = [C.c_int, C.c_size_t, C.POINTER(C.c_void_p)]
        L.h2v_dev_alloc.argtypes = [C.c_size_t, C.POINTER(C.c_void_p)]
        L.h2v_dev_free.argtypes = [C.c_void_p]
        L.h2v_dev_upload.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.h2v_dev_download.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.h2v_host_register.argtypes = [C.c_void_p, C.c_size_t]
        L.h2v_host_unregister.argtypes = [C.c_void_p]
        L.h2v_srs_load.argtypes = [C.c_uint32, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]
        L.h2v_srs_setup.argtypes = [C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]
        L.h2v_srs_free.argtypes = [C.c_void_p]
        L.h2v_srs_info.argtypes = [C.c_void_p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
        L.h2v_srs_free.restype = None
        L.h2v_commit.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]
        L.h2v_commit_batch.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.c_size_t, C.c_size_t, C.c_void_p]
        L.h2v_commit_batch_dev.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_void_p]
        L.h2v_best_multiexp.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        L.h2v_g1_sum.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p]
        L.h2v_best_fft.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
        L.h2v_domain_new.argtypes = [C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p)]
        L.h2v_domain_free.argtypes = [C.c_void_p]
        L.h2v_domain_free.restype = None
        L.h2v_domain_constant.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        for name in ("h2v_lagrange_to_coeff", "h2v_coeff_to_lagrange", "h2v_divide_by_vanishing_poly"):
            getattr(L, name).argtypes = [C.c_void_p, C.c_void_p]
        for name in ("h2v_coeff_to_extended", "h2v_extended_to_coeff"):
            getattr(L, name).argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.h2v_domain_transform_batch.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_size_t]
        L.h2v_domain_transform_dev.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_size_t]
        L.h2v_eval_polynomial_batch.argtypes = [C.POINTER(C.c_void_p), C.c_size_t, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]
        L.h2v_eval_polynomial_dev.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]
        L.h2v_batch_invert.argtypes = [C.c_void_p, C.c_size_t]
        L.h2v_grand_product.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        L.h2v_grand_product_dev.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p]
        L.h2v_kate_division.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
        L.h2v_permute_expression_pair.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
        L.h2v_permute_expression_pair_dev.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
        L.h2v_permute_expression_pair_batch_dev.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
        L.h2v_quotient_gates_dev.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
        L.h2v_quotient_permutation_dev.argtypes = ([C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t]
                                                   + [C.c_void_p, C.c_size_t] * 3 + [C.c_void_p] * 3 + [C.c_uint32])
        L.h2v_quotient_lookup_dev.argtypes = [C.c_void_p] * 13
        L.h2v_g1_to_bytes.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p]
        L.h2v_fr_to_repr.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p]
        L.h2v_commit_batch_resident.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_size_t, C.c_size_t,
                                                C.c_void_p, C.c_size_t, C.c_void_p]
        L.h2v_selftest_field.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        L.h2v_selftest_group.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        L.h2v_synthetic_bases.argtypes = [C.c_uint64, C.c_uint64, C.c_size_t, C.c_void_p]
        L.h2v_selftest_imad_peak.argtypes = [C.POINTER(C.c_double)]
        L.h2v_selftest_imad_probe.argtypes = [C.c_int, C.POINTER(C.c_double)]
        L.h2v_selftest_op_rate.argtypes = [C.c_int, C.POINTER(C.c_double)]
        L.h2v_set_tuning.argtypes = [C.c_int, C.c_int]
        L.h2v_last_kernel_ms.argtypes = [C.POINTER(C.c_float)]
        L.h2v_last_msm_entries.restype = C.c_uint64
        L.h2v_domain_rotate_omega.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
        L.h2v_domain_rotate_extended.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
        L.h2v_domain_l_i_range.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]
        L.h2v_domain_fill.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.h2v_kate_division_dev.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
        L.h2v_quotient_gates_ptrs_dev.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
        L.h2v_quotient_permutation_ptrs_dev.argtypes = ([C.c_void_p] * 5 + [C.c_size_t, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p,
                                                        C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32])
        L.h2v_quotient_permutation_range_ptrs_dev.argtypes = ([C.c_void_p] * 5 + [C.c_size_t] * 4 + [C.c_int]
                                                              + [C.c_void_p] * 3 + [C.c_size_t] + [C.c_void_p] * 3 + [C.c_uint32])
        L.h2v_pk_load.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_void_p, C.POINTER(C.c_void_p)]
        L.h2v_pk_free.argtypes = [C.c_void_p]
        L.h2v_pk_free.restype = None
        L.h2v_create_proof.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_size_t, C.POINTER(C.c_size_t)]
        L.h2v_create_proofs.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_char_p,
                                        C.c_void_p, C.c_size_t]
        L.h2v_proof_size.argtypes = [C.c_void_p]
        L.h2v_proof_size.restype = C.c_size_t
        L.h2v_pk_last_phase_ms.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
        L.h2v_mock_prover.argtypes = [C.c_void_p] * 7 + [C.c_size_t, C.POINTER(C.c_uint64)]
        L.h2v_pk_mock_prover.argtypes = [C.c_void_p, C.c_size_t] + [C.c_void_p] * 4 + [C.c_size_t, C.c_void_p]
        L.h2v_mock_last_ms.argtypes = [C.POINTER(C.c_double)]
        L.h2v_create_proofs_from_inputs.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_char_p, C.c_void_p,
                                                    C.c_size_t, C.c_void_p]
        L.h2v_pk_mock_prover_from_inputs.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_void_p, C.c_size_t,
                                                     C.c_void_p]
        L.h2v_transcript_new.argtypes = [C.POINTER(C.c_void_p)]
        L.h2v_transcript_free.argtypes = [C.c_void_p]
        L.h2v_transcript_free.restype = None
        for name in ("common_point", "common_scalar", "write_point", "write_scalar", "squeeze_challenge"):
            getattr(L, "h2v_transcript_" + name).argtypes = [C.c_void_p, C.c_void_p]
        L.h2v_transcript_bytes.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
        L.h2v_poseidon_permutation.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]
        L.h2v_poseidon_permutation_variant.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p]
        L.h2v_chacha20_fr_random.argtypes = [C.c_char_p, C.c_size_t, C.c_void_p]
        L.h2v_chacha20_block.argtypes = [C.c_char_p, C.c_uint64, C.c_void_p]
        L.h2v_srs_gen.argtypes = [C.c_uint32, C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.h2v_g2_mul_generator.argtypes = [C.c_void_p, C.c_void_p]
        L.h2v_srs_write_file.argtypes = [C.c_char_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.h2v_srs_read_file.argtypes = [C.c_char_p, C.POINTER(C.c_uint32), C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def _check(rc):
    if rc != 0:
        msg = lib().h2v_last_error().decode(errors="replace")
        if rc == -1:
            raise ValueError(msg)      # upstream: assert!/panic on a malformed argument
        raise H2VError(msg)            # CUDA failure: hard error, never a fallback


def _fr(a, n=None):
    a = np.ascontiguousarray(a, dtype=np.uint64)
    if a.ndim != 2 or a.shape[1] != 4 or (n is not None and a.shape[0] != n):
        raise ValueError(f"expected Fr array of shape ({'n' if n is None else n}, 4), got {a.shape}")
    return a


def _fr1(x):
    return _fr(np.asarray(x, dtype=np.uint64).reshape(1, 4), 1)


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def init(devices=0):
    """`h2v_init(devices, n_dev)`: the CUDA device(s) this process drives -- an int or a list; the first one is the primary
    device.  With several devices every handle holds a replica per device and the host-facing batch entry points split
    their columns across them (column j -> device j mod G)."""
    devs = [int(devices)] if isinstance(devices, (int, np.integer)) else [int(d) for d in devices]
    arr = (C.c_int * len(devs))(*devs)
    _check(lib().h2v_init(arr, len(devs)))


def device_list():
    buf = (C.c_int * 16)()
    n = lib().h2v_device_list(buf, 16)
    return [int(buf[i]) for i in range(n)]


class DeviceBuffer:
    """A device allocation for the `_dev` entry points (columns resident in HBM across several steps)."""

    def __init__(self, nbytes, device=None):
        self.nbytes = nbytes
        self._p = C.c_void_p()
        if device is None:
            _check(lib().h2v_dev_alloc(nbytes, C.byref(self._p)))
        else:
            _check(lib().h2v_dev_alloc_on(device, nbytes, C.byref(self._p)))

    @property
    def ptr(self):
        return self._p.value

    def upload(self, arr, offset=0):
        arr = np.ascontiguousarray(arr)
        if offset + arr.nbytes > self.nbytes:
            raise ValueError("upload out of range")
        _check(lib().h2v_dev_upload(self._p.value + offset, arr.ctypes.data_as(C.c_void_p), arr.nbytes))

    def download(self, shape, dtype=np.uint64, offset=0):
        out = np.zeros(shape, dtype=dtype)
        if offset + out.nbytes > self.nbytes:
            raise ValueError("download out of range")
        _check(lib().h2v_dev_download(out.ctypes.data_as(C.c_void_p), self._p.value + offset, out.nbytes))
        return out

    def free(self):
        if self._p.value and _lib is not None:
            _lib.h2v_dev_free(self._p)
            self._p = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def host_register(arr):
    """Page-lock a numpy array in place (faster, overlappable copies through the host-facing entry points)."""
    _check(lib().h2v_host_register(arr.ctypes.data_as(C.c_void_p), arr.nbytes))


def host_unregister(arr):
    _check(lib().h2v_host_unregister(arr.ctypes.data_as(C.c_void_p)))


def device_count():
    return lib().h2v_device_count()


def launch_count():
    return int(lib().h2v_launch_count())


def last_kernel_ms():
    buf = (C.c_float * 8)()
    _check(lib().h2v_last_kernel_ms(buf))
    return dict(zip(KERNEL_CLASSES, [float(x) for x in buf]))


def last_msm_entries():
    """mixed additions (non-zero digits) the calling thread's last commit_batch_dev executed"""
    return int(lib().h2v_last_msm_entries())


def imad_peak():
    out = C.c_double()
    _check(lib().h2v_selftest_imad_peak(C.byref(out)))
    return out.value


def imad_probe(which=1):
    """IMAD.WIDE.U32 issue rate (wide multiply-adds per second): 0 = round-1 probe, 1 = pure chain probe"""
    out = C.c_double()
    _check(lib().h2v_selftest_imad_probe(which, C.byref(out)))
    return out.value


def set_tuning(chunk=-1, table=-1):
    """MSM tuning knobs (-1 = automatic): results never depend on them."""
    _check(lib().h2v_set_tuning(chunk, table))


def op_rate(which):
    """0: Fq mul/s (1 chain per thread), 1: Fq mul/s (2 chains), 2: XYZZ mixed adds/s -- registers only."""
    out = C.c_double()
    _check(lib().h2v_selftest_op_rate(which, C.byref(out)))
    return out.value


# ----------------------------------------------------------------------------- arithmetic.rs
def best_multiexp(coeffs, bases):
    """halo2-axiom arithmetic.rs `best_multiexp(coeffs, bases) -> C::Curve` (Jacobian, 12 limbs)."""
    coeffs = _fr(coeffs)
    bases = np.ascontiguousarray(bases, dtype=np.uint64)
    if bases.ndim != 2 or bases.shape[1] != 8:
        raise ValueError(f"expected G1Affine array of shape (n, 8), got {bases.shape}")
    if coeffs.shape[0] != bases.shape[0]:
        raise ValueError("best_multiexp: assertion failed: coeffs.len() == bases.len()")
    out = np.zeros(12, dtype=np.uint64)
    _check(lib().h2v_best_multiexp(_ptr(coeffs), _ptr(bases), coeffs.shape[0], _ptr(out)))
    return out


def g1_sum(points):
    """Sum of affine points -> affine (combines the per-GPU partial sums of a multiexp split by index range)."""
    pts = np.ascontiguousarray(points, dtype=np.uint64).reshape(-1, 8)
    out = np.zeros(8, dtype=np.uint64)
    _check(lib().h2v_g1_sum(_ptr(pts), pts.shape[0], _ptr(out)))
    return out


def best_fft(a, omega, log_n):
    """halo2-axiom arithmetic.rs `best_fft(a, omega, log_n)`; returns the transformed copy."""
    a = np.array(_fr(a), copy=True)
    if a.shape[0] != 1 << log_n:
        raise ValueError("best_fft: assertion failed: a.len() == 1 << log_n")
    omega = np.ascontiguousarray(omega, dtype=np.uint64).reshape(4)
    _check(lib().h2v_best_fft(_ptr(a), _ptr(omega), log_n))
    return a


def eval_polynomial(poly, point):
    """halo2-axiom arithmetic.rs `eval_polynomial(poly, point)` (Horner) -> (4,)"""
    return eval_polynomial_batch([poly], np.ascontiguousarray(point, dtype=np.uint64).reshape(1, 4))[0, 0]


def eval_polynomial_batch(polys, points):
    """every polynomial at every point -> (n_polys, n_points, 4)"""
    cols = [_fr(p) for p in polys]
    points = _fr(points)
    out = np.zeros((len(cols), points.shape[0], 4), dtype=np.uint64)
    if cols and points.shape[0]:
        ln = cols[0].shape[0]
        if any(c.shape[0] != ln for c in cols):
            raise ValueError("eval_polynomial_batch: polynomials must have equal length")
        arr = (C.c_void_p * len(cols))(*[c.ctypes.data for c in cols])
        _check(lib().h2v_eval_polynomial_batch(arr, len(cols), ln, _ptr(points), points.shape[0], _ptr(out)))
    return out


def batch_invert(a):
    """ff `BatchInvert::batch_invert`: non-zero elements inverted, zeros untouched (returns a copy)."""
    a = np.array(_fr(a), copy=True)
    _check(lib().h2v_batch_invert(_ptr(a), a.shape[0]))
    return a


def grand_product(num, den):
    """z[0] = 1, z[i+1] = z[i] * num[i] / den[i]: the running product of the permutation / lookup arguments."""
    num, den = _fr(num), _fr(den)
    if num.shape != den.shape:
        raise ValueError("grand_product: num and den must have equal length")
    out = np.zeros_like(num)
    _check(lib().h2v_grand_product(_ptr(num), _ptr(den), num.shape[0], _ptr(out)))
    return out


def grand_product_dev(d_num, d_den, n, n_cols, d_out):
    """Running products of n_cols contiguous device-resident columns (one batch inversion for all)."""
    _check(lib().h2v_grand_product_dev(d_num, d_den, n, n_cols, d_out))


def kate_division_dev(d_a, n, b, d_out):
    _check(lib().h2v_kate_division_dev(d_a, n, _ptr(_fr1(b)), d_out))


def kate_division(a, b):
    """halo2-axiom arithmetic.rs `kate_division(a, b)`: quotient of a(X) by (X - b)."""
    a = _fr(a)
    out = np.zeros((max(a.shape[0] - 1, 0), 4), dtype=np.uint64)
    b = np.ascontiguousarray(b, dtype=np.uint64).reshape(4)
    _check(lib().h2v_kate_division(_ptr(a), a.shape[0], _ptr(b), _ptr(out)))
    return out


def permute_expression_pair(inp, table):
    """plonk/lookup/prover.rs permute_expression_pair on the usable rows -> (permuted_input, permuted_table)."""
    inp, table = _fr(inp), _fr(table)
    if inp.shape != table.shape:
        raise ValueError("input and table must have the same number of usable rows")
    a, s = np.zeros_like(inp), np.zeros_like(inp)
    _check(lib().h2v_permute_expression_pair(_ptr(inp), _ptr(table), inp.shape[0], _ptr(a), _ptr(s)))
    return a, s


def permute_expression_pair_batch_dev(d_inputs, d_tables, usable_rows, d_permuted_inputs, input_stride, d_permuted_tables, table_stride):
    """all lookups of a phase at once: lists of device column pointers in, strided device output matrices"""
    L = len(d_inputs)
    ia = (C.c_void_p * max(1, L))(*d_inputs)
    ta = (C.c_void_p * max(1, L))(*d_tables)
    _check(lib().h2v_permute_expression_pair_batch_dev(ia, ta, L, usable_rows, d_permuted_inputs, input_stride, d_permuted_tables, table_stride))


def permute_expression_pair_dev(d_input, d_table, usable_rows, d_permuted_input, d_permuted_table):
    _check(lib().h2v_permute_expression_pair_dev(d_input, d_table, usable_rows, d_permuted_input, d_permuted_table))


def g1_to_bytes(points):
    """halo2curves `G1Affine::to_bytes()` for (n, 8) affine points -> list of 32-byte strings (host-side)."""
    pts = np.ascontiguousarray(points, dtype=np.uint64).reshape(-1, 8)
    out = np.zeros((pts.shape[0], 32), dtype=np.uint8)
    _check(lib().h2v_g1_to_bytes(_ptr(pts), pts.shape[0], _ptr(out)))
    return [bytes(r) for r in out]


def fr_to_repr(scalars):
    """`Fr::to_repr()` for (n, 4) Montgomery scalars -> list of 32-byte little-endian strings (host-side)."""
    a = _fr(scalars)
    out = np.zeros((a.shape[0], 32), dtype=np.uint8)
    _check(lib().h2v_fr_to_repr(_ptr(a), a.shape[0], _ptr(out)))
    return [bytes(r) for r in out]


# ----------------------------------------------------------------------------- poly/kzg/commitment.rs
def srs_setup(k, s):
    """`ParamsKZG::setup(k, rng)` with the secret s (Montgomery Fr, (4,)) given: returns (g, g_lagrange)."""
    n = 1 << k
    s = np.ascontiguousarray(s, dtype=np.uint64).reshape(4)
    g = np.zeros((n, 8), dtype=np.uint64)
    gl = np.zeros((n, 8), dtype=np.uint64)
    _check(lib().h2v_srs_setup(k, _ptr(s), _ptr(g), _ptr(gl)))
    return g, gl


def g2_mul_generator(s):
    """s * G2 generator as a raw G2Affine (16 limbs: x.c0, x.c1, y.c0, y.c1 Montgomery); host-side"""
    out = np.zeros(16, dtype=np.uint64)
    _check(lib().h2v_g2_mul_generator(_ptr(_fr1(s)), _ptr(out)))
    return out


def gen_srs_secret(seed=bytes(32)):
    """the setup secret of `ParamsKZG::setup(k, ChaCha20Rng::from_seed(seed))` (gen_srs: seed of zeros), Montgomery (4,)"""
    return chacha20_fr_random(seed, 1)[0]


def write_srs(path, k, g, g_lagrange, g2, s_g2):
    """`ParamsKZG::write` (RawBytes) -- the reference's params/kzg_bn254_{k}.srs"""
    g = np.ascontiguousarray(g, dtype=np.uint64).reshape(1 << k, 8)
    gl = np.ascontiguousarray(g_lagrange, dtype=np.uint64).reshape(1 << k, 8)
    _check(lib().h2v_srs_write_file(os.fsencode(path), k, _ptr(g), _ptr(gl), _ptr(np.ascontiguousarray(g2, dtype=np.uint64).reshape(16)),
                                    _ptr(np.ascontiguousarray(s_g2, dtype=np.uint64).reshape(16))))


def read_srs(path):
    """`ParamsKZG::read` -> (k, g, g_lagrange, g2, s_g2)"""
    k = C.c_uint32()
    lib().h2v_srs_read_file(os.fsencode(path), C.byref(k), None, None, 0, None, None)      # header only
    if k.value == 0 and not os.path.exists(path):
        raise ValueError(f"cannot open {path}")
    n = 1 << k.value
    g, gl = np.zeros((n, 8), dtype=np.uint64), np.zeros((n, 8), dtype=np.uint64)
    g2, sg2 = np.zeros(16, dtype=np.uint64), np.zeros(16, dtype=np.uint64)
    _check(lib().h2v_srs_read_file(os.fsencode(path), C.byref(k), _ptr(g), _ptr(gl), n, _ptr(g2), _ptr(sg2)))
    return k.value, g, gl, g2, sg2


class ParamsKZG:
    """halo2-axiom `ParamsKZG<Bn256>` restricted to the commit path: {k, n, g, g_lagrange}."""

    def __init__(self, k, g=None, g_lagrange=None):
        self.k, self.n = k, 1 << k
        self._h = C.c_void_p()
        ptrs = []
        for b in (g, g_lagrange):
            if b is None:
                ptrs.append(None)
                continue
            b = np.ascontiguousarray(b, dtype=np.uint64)
            if b.shape != (self.n, 8):
                raise ValueError(f"expected ({self.n}, 8) G1Affine bases, got {b.shape}")
            ptrs.append(b)
        _check(lib().h2v_srs_load(k, None if ptrs[0] is None else _ptr(ptrs[0]),
                                  None if ptrs[1] is None else _ptr(ptrs[1]), C.byref(self._h)))

    @classmethod
    def setup(cls, k, s):
        """`ParamsKZG::setup`: build both bases on the device from the secret s and load them."""
        g, gl = srs_setup(k, s)
        p = cls(k, g, gl)
        p.g, p.g_lagrange = g, gl
        return p

    @classmethod
    def gen_srs(cls, k, seed=bytes(32), params_dir=None):
        """halo2-base `gen_srs(k)` (scaffold mod.rs:260): read `params_dir/kzg_bn254_{k}.srs` if it exists, else run the
        seeded setup (seed of zeros upstream) on the device and write the file; the bases are loaded either way."""
        path = None if params_dir is None else os.path.join(params_dir, f"kzg_bn254_{k}.srs")
        if path and os.path.exists(path):
            fk, g, gl, g2, sg2 = read_srs(path)
            if fk != k:
                raise ValueError(f"{path} holds k = {fk}")
        else:
            n = 1 << k
            g, gl = np.zeros((n, 8), dtype=np.uint64), np.zeros((n, 8), dtype=np.uint64)
            g2, sg2 = np.zeros(16, dtype=np.uint64), np.zeros(16, dtype=np.uint64)
            _check(lib().h2v_srs_gen(k, bytes(seed), _ptr(g), _ptr(gl), _ptr(g2), _ptr(sg2)))
            if path:
                os.makedirs(params_dir, exist_ok=True)
                write_srs(path, k, g, gl, g2, sg2)
        p = cls(k, g, gl)
        p.g, p.g_lagrange, p.g2, p.s_g2 = g, gl, g2, sg2
        return p

    def close(self):
        if getattr(self, "_h", None) and self._h.value and _lib is not None:
            _lib.h2v_srs_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:      # interpreter shutdown: module globals may already be gone
            pass

    def info(self):
        """(window bits c, windows W) of the precomputed tables."""
        c, w = C.c_uint32(), C.c_uint32()
        _check(lib().h2v_srs_info(self._h, C.byref(c), C.byref(w)))
        return c.value, w.value

    def _commit(self, basis, poly):
        poly = _fr(poly)
        out = np.zeros(8, dtype=np.uint64)
        _check(lib().h2v_commit(self._h, basis, _ptr(poly), poly.shape[0], _ptr(out)))
        return out

    def commit(self, poly, blind=None):
        """`commit(&poly, _blind)`: monomial basis; the blind is ignored by KZG upstream. Affine (8,)."""
        return self._commit(H2V_BASIS_MONOMIAL, poly)

    def commit_lagrange(self, poly, blind=None):
        return self._commit(H2V_BASIS_LAGRANGE, poly)

    def commit_batch(self, polys, basis=H2V_BASIS_LAGRANGE):
        """Commit a list of equal-length columns against one basis in a single call -> (n_polys, 8)."""
        cols = [_fr(p) for p in polys]
        if not cols:
            return np.zeros((0, 8), dtype=np.uint64)
        ln = cols[0].shape[0]
        if any(c.shape[0] != ln for c in cols):
            raise ValueError("commit_batch: columns must have equal length")
        arr = (C.c_void_p * len(cols))(*[c.ctypes.data for c in cols])
        out = np.zeros((len(cols), 8), dtype=np.uint64)
        _check(lib().h2v_commit_batch(self._h, basis, arr, len(cols), ln, _ptr(out)))
        return out

    def commit_batch_resident(self, polys, tails, row0, d_dst_ptr, dst_stride, basis=H2V_BASIS_LAGRANGE):
        """Host columns committed AND left resident at d_dst (one of the h2v_init devices); rows row0.. of column j are
        overwritten with tails[j] (shape (n_polys, n_rows, 4), the blinding rows of create_proof) before the commit."""
        polys = [np.ascontiguousarray(p, dtype=np.uint64) for p in polys]
        n_polys, length = len(polys), (polys[0].shape[0] if polys else 0)
        tails = np.ascontiguousarray(tails, dtype=np.uint64) if tails is not None else None
        n_rows = 0 if tails is None else tails.shape[1]
        arr = (C.c_void_p * max(1, n_polys))(*[p.ctypes.data for p in polys])
        out = np.zeros((n_polys, 8), dtype=np.uint64)
        _check(lib().h2v_commit_batch_resident(self._h, basis, arr, n_polys, length, _ptr(tails) if n_rows else None, row0, n_rows,
                                               C.c_void_p(d_dst_ptr), dst_stride, _ptr(out)))
        return out

    def commit_batch_dev(self, d_polys_ptr, col_stride, n_polys, length, d_out_ptr, basis=H2V_BASIS_LAGRANGE):
        """Device-resident columns (raw device pointers, e.g. torch tensor .data_ptr())."""
        _check(lib().h2v_commit_batch_dev(self._h, basis, d_polys_ptr, col_stride, n_polys, length, d_out_ptr))


# ----------------------------------------------------------------------------- poly/domain.rs
class EvaluationDomain:
    """halo2-axiom `EvaluationDomain::new(j, k)` and its transforms."""

    _CONST = ["omega", "omega_inv", "extended_omega", "extended_omega_inv", "g_coset", "g_coset_inv",
              "ifft_divisor", "extended_ifft_divisor"]

    def __init__(self, j, k):
        self._h = C.c_void_p()
        _check(lib().h2v_domain_new(j, k, C.byref(self._h)))
        self.j, self.k, self.n = j, k, 1 << k
        self.extended_k = int(lib().h2v_domain_extended_k(self._h))
        self.extended_n = 1 << self.extended_k
        for i, name in enumerate(self._CONST):
            setattr(self, name, self._constant(i))
        self.t_evaluations = [self._constant(8 + i) for i in range(1 << (self.extended_k - k))]

    def _constant(self, which):
        out = np.zeros(4, dtype=np.uint64)
        _check(lib().h2v_domain_constant(self._h, which, _ptr(out)))
        return out

    def close(self):
        if getattr(self, "_h", None) and self._h.value and _lib is not None:
            _lib.h2v_domain_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def get_quotient_poly_degree(self):
        return self.j - 1

    def lagrange_to_coeff(self, a):
        a = np.array(_fr(a, self.n), copy=True)
        _check(lib().h2v_lagrange_to_coeff(self._h, _ptr(a)))
        return a

    def coeff_to_lagrange(self, a):
        a = np.array(_fr(a, self.n), copy=True)
        _check(lib().h2v_coeff_to_lagrange(self._h, _ptr(a)))
        return a

    def coeff_to_extended(self, a):
        a = _fr(a, self.n)
        out = np.zeros((self.extended_n, 4), dtype=np.uint64)
        _check(lib().h2v_coeff_to_extended(self._h, _ptr(a), _ptr(out)))
        return out

    def extended_to_coeff(self, a):
        a = _fr(a, self.extended_n)
        out = np.zeros((self.n * (self.j - 1), 4), dtype=np.uint64)
        _check(lib().h2v_extended_to_coeff(self._h, _ptr(a), _ptr(out)))
        return out

    def divide_by_vanishing_poly(self, a):
        a = np.array(_fr(a, self.extended_n), copy=True)
        _check(lib().h2v_divide_by_vanishing_poly(self._h, _ptr(a)))
        return a

    def transform_batch(self, op, cols):
        """One EvaluationDomain op over a list of independent columns (host arrays) -> list of arrays."""
        nin = self.extended_n if op in (OP_EXTENDED_TO_COEFF, OP_DIVIDE_BY_VANISHING) else self.n
        nout = (self.extended_n if op == OP_COEFF_TO_EXTENDED else
                self.n * (self.j - 1) if op in (OP_EXTENDED_TO_COEFF, OP_DIVIDE_BY_VANISHING) else self.n)
        ins = [_fr(c, nin) for c in cols]
        outs = [np.zeros((nout, 4), dtype=np.uint64) for _ in ins]
        if ins:
            ia = (C.c_void_p * len(ins))(*[c.ctypes.data for c in ins])
            oa = (C.c_void_p * len(ins))(*[c.ctypes.data for c in outs])
            _check(lib().h2v_domain_transform_batch(self._h, op, ia, oa, len(ins)))
        return outs

    def transform_dev(self, op, d_in_ptr, in_stride, d_out_ptr, out_stride, n_cols):
        _check(lib().h2v_domain_transform_dev(self._h, op, d_in_ptr, in_stride, d_out_ptr, out_stride, n_cols))

    # --- evaluate_h row loops on device-resident extended columns (halo2-axiom plonk/evaluation.rs [UPSTREAM])
    def quotient_gates(self, d_h, y, n_gates, d_q, q_stride, d_a, a_stride):
        """h <- h*y + q_j*(a_j + a_j(wX)*a_j(w^2X) - a_j(w^3X)) for every halo2-base vertical gate j, in order."""
        _check(lib().h2v_quotient_gates_dev(self._h, d_h, _ptr(_fr1(y)), n_gates, d_q, q_stride, d_a, a_stride))

    def quotient_permutation(self, d_h, y, beta, gamma, n_cols, chunk_len, d_cols, cols_stride, d_sigma, sigma_stride,
                             d_z, z_stride, d_l0, d_l_last, d_l_active, blinding_factors):
        _check(lib().h2v_quotient_permutation_dev(self._h, d_h, _ptr(_fr1(y)), _ptr(_fr1(beta)), _ptr(_fr1(gamma)),
                                                  n_cols, chunk_len, d_cols, cols_stride, d_sigma, sigma_stride, d_z, z_stride,
                                                  d_l0, d_l_last, d_l_active, blinding_factors))

    def quotient_permutation_range(self, d_h, y, beta, gamma, n_cols, chunk_len, set_begin, set_end, with_head, d_col_ptrs,
                                   d_sigma_ptrs, d_z, z_stride, d_l0, d_l_last, d_l_active, blinding_factors):
        """The permutation terms of the sets [set_begin, set_end) only (a prover that streams the extended columns through
        HBM in slices).  d_col_ptrs / d_sigma_ptrs are device tables of column pointers whose entry 0 is column
        set_begin * chunk_len; d_z holds all the sets' z columns.  `with_head` folds the terms that precede the per-set
        products: set it on the first call only, and consecutive ranges fold to the result of one quotient_permutation."""
        _check(lib().h2v_quotient_permutation_range_ptrs_dev(self._h, d_h, _ptr(_fr1(y)), _ptr(_fr1(beta)), _ptr(_fr1(gamma)), n_cols,
                                                             chunk_len, set_begin, set_end, int(bool(with_head)), d_col_ptrs,
                                                             d_sigma_ptrs, d_z, z_stride, d_l0, d_l_last, d_l_active, blinding_factors))

    def quotient_lookup(self, d_h, y, beta, gamma, d_input, d_table, d_perm_input, d_perm_table, d_z, d_l0, d_l_last, d_l_active):
        _check(lib().h2v_quotient_lookup_dev(self._h, d_h, _ptr(_fr1(y)), _ptr(_fr1(beta)), _ptr(_fr1(gamma)),
                                             d_input, d_table, d_perm_input, d_perm_table, d_z, d_l0, d_l_last, d_l_active))


    # --- scalar / index helpers of poly/domain.rs (host-side)
    def rotate_omega(self, value, rotation):
        """`rotate_omega(value, Rotation(rotation))` = value * omega^rotation"""
        out = np.zeros(4, dtype=np.uint64)
        _check(lib().h2v_domain_rotate_omega(self._h, _ptr(_fr1(value)), rotation, _ptr(out)))
        return out

    def rotate_extended(self, poly, rotation):
        """`rotate_extended(&poly, Rotation(rotation))` on an extended-domain column (returns a new array)"""
        a = _fr(poly, self.extended_n)
        out = np.zeros_like(a)
        _check(lib().h2v_domain_rotate_extended(self._h, _ptr(a), rotation, _ptr(out)))
        return out

    def l_i_range(self, x, xn, rotations):
        """`l_i_range(x, xn, rotations)` for a contiguous `range(lo, hi)` of rotations -> (hi - lo, 4)"""
        rot = list(rotations)
        if rot != list(range(rot[0], rot[0] + len(rot))) if rot else False:
            raise ValueError("l_i_range: rotations must be a contiguous ascending range")
        out = np.zeros((len(rot), 4), dtype=np.uint64)
        if rot:
            _check(lib().h2v_domain_l_i_range(self._h, _ptr(_fr1(x)), _ptr(_fr1(xn)), rot[0], rot[0] + len(rot), _ptr(out)))
        return out

    def _fill(self, basis, scalar):
        out = np.zeros((self.extended_n if basis == 2 else self.n, 4), dtype=np.uint64)
        _check(lib().h2v_domain_fill(self._h, basis, None if scalar is None else _ptr(_fr1(scalar)), _ptr(out)))
        return out

    def empty_coeff(self):
        return self._fill(0, None)

    def empty_lagrange(self):
        return self._fill(1, None)

    def empty_extended(self):
        return self._fill(2, None)

    def constant_lagrange(self, scalar):
        return self._fill(1, scalar)

    def constant_extended(self, scalar):
        return self._fill(2, scalar)

    def extended_len(self):
        return self.extended_n

    def get_omega(self):
        return self.omega

    def get_omega_inv(self):
        return self.omega_inv

    def get_extended_omega(self):
        return self.extended_omega


# ----------------------------------------------------------------------------- transcript / RNG (host-side)
class PoseidonTranscript:
    """snark-verifier `PoseidonTranscript<G1Affine, NativeLoader, Vec<u8>, 5, 4, 8, 60>::new::<0>` (writer)."""

    def __init__(self):
        self._h = C.c_void_p()
        _check(lib().h2v_transcript_new(C.byref(self._h)))

    def __del__(self):
        try:
            if self._h.value and _lib is not None:
                _lib.h2v_transcript_free(self._h)
                self._h = C.c_void_p()
        except Exception:
            pass

    def _pt(self, p):
        return _ptr(np.ascontiguousarray(p, dtype=np.uint64).reshape(8))

    def common_point(self, p):
        _check(lib().h2v_transcript_common_point(self._h, self._pt(p)))

    def common_scalar(self, s):
        _check(lib().h2v_transcript_common_scalar(self._h, _ptr(_fr1(s))))

    def write_point(self, p):
        _check(lib().h2v_transcript_write_point(self._h, self._pt(p)))

    def write_scalar(self, s):
        _check(lib().h2v_transcript_write_scalar(self._h, _ptr(_fr1(s))))

    def squeeze_challenge(self):
        out = np.zeros(4, dtype=np.uint64)
        _check(lib().h2v_transcript_squeeze_challenge(self._h, _ptr(out)))
        return out

    def finalize(self):
        ln = C.c_size_t()
        _check(lib().h2v_transcript_bytes(self._h, None, 0, C.byref(ln)))
        buf = np.zeros(max(ln.value, 1), dtype=np.uint8)
        _check(lib().h2v_transcript_bytes(self._h, _ptr(buf), ln.value, C.byref(ln)))
        return bytes(buf[:ln.value])


def poseidon_permutation(state, r_f, r_p, variant=1):
    """the Poseidon permutation over BN254 Fr (t = len(state) in {3, 5}) on Montgomery-form words; returns a new array.
    variant 0 = plain rounds, 1 = the sparse form the transcript uses (identical results)"""
    st = np.array(_fr(state), copy=True)
    _check(lib().h2v_poseidon_permutation_variant(st.shape[0], r_f, r_p, variant, _ptr(st)))
    return st


def chacha20_fr_random(seed, n):
    """the first n `Fr::random(&mut ChaCha20Rng::from_seed(seed))` draws, Montgomery form (n, 4)"""
    out = np.zeros((n, 4), dtype=np.uint64)
    _check(lib().h2v_chacha20_fr_random(bytes(seed), n, _ptr(out)))
    return out


def chacha20_block(seed, counter):
    out = np.zeros(64, dtype=np.uint8)
    _check(lib().h2v_chacha20_block(bytes(seed), counter, _ptr(out)))
    return bytes(out)


# ----------------------------------------------------------------------------- plonk/prover.rs
class _CircuitT(C.Structure):
    _fields_ = [("k", C.c_uint32), ("degree", C.c_uint32), ("blinding_factors", C.c_uint32),
                ("n_advice", C.c_uint32), ("n_fixed", C.c_uint32), ("n_instance", C.c_uint32),
                ("n_gates", C.c_uint32), ("gate_advice", C.c_void_p), ("gate_selector", C.c_void_p),
                ("n_lookups", C.c_uint32), ("lookup_input", C.c_void_p), ("lookup_table", C.c_void_p),
                ("n_perm", C.c_uint32), ("perm_kind", C.c_void_p), ("perm_index", C.c_void_p),
                ("n_advice_queries", C.c_uint32), ("advice_query_col", C.c_void_p), ("advice_query_rot", C.c_void_p),
                ("n_fixed_queries", C.c_uint32), ("fixed_query_col", C.c_void_p), ("fixed_query_rot", C.c_void_p)]


def _circuit_struct(cs):
    """cs dict (see ProvingKey) -> (h2v_circuit_t, the index arrays it points into: keep them alive while it is used)"""
    u32 = lambda xs: np.ascontiguousarray(xs, dtype=np.uint32)
    a = dict(
        ga=u32([g[0] for g in cs["gates"]]), gs=u32([g[1] for g in cs["gates"]]),
        li=u32([l[0] for l in cs["lookups"]]), lt=u32([l[1] for l in cs["lookups"]]),
        pk=np.ascontiguousarray([p[0] for p in cs["permutation"]], dtype=np.uint8), pi=u32([p[1] for p in cs["permutation"]]),
        aqc=u32([q[0] for q in cs["advice_queries"]]), aqr=np.ascontiguousarray([q[1] for q in cs["advice_queries"]], dtype=np.int32),
        fqc=u32([q[0] for q in cs["fixed_queries"]]), fqr=np.ascontiguousarray([q[1] for q in cs["fixed_queries"]], dtype=np.int32))
    p = lambda x: x.ctypes.data if x.size else None
    ct = _CircuitT(cs["k"], cs["degree"], cs["blinding_factors"], cs["n_advice"], cs["n_fixed"], cs["n_instance"],
                   len(cs["gates"]), p(a["ga"]), p(a["gs"]), len(cs["lookups"]), p(a["li"]), p(a["lt"]),
                   len(cs["permutation"]), p(a["pk"]), p(a["pi"]), len(cs["advice_queries"]), p(a["aqc"]), p(a["aqr"]),
                   len(cs["fixed_queries"]), p(a["fqc"]), p(a["fqr"]))
    return ct, a


class ProvingKey:
    """halo2 `ProvingKey` for a halo2-base-shaped constraint system, resident on the device.

    cs: dict with k, degree, blinding_factors, n_advice, n_fixed, n_instance, gates [(advice, selector)],
    lookups [(input advice, table fixed)], permutation [(kind, index)] (kind 0 advice, 1 fixed, 2 instance),
    advice_queries [(column, rotation)], fixed_queries [(column, rotation)]."""

    def __init__(self, params, cs, fixed, sigma, vk_transcript_repr):
        self.params, self.cs = params, cs
        ct, self._arrs = _circuit_struct(cs)
        n = 1 << cs["k"]
        fx = [_fr(c, n) for c in fixed]
        sg = [_fr(c, n) for c in sigma]
        if len(fx) != cs["n_fixed"] or len(sg) != len(cs["permutation"]):
            raise ValueError("ProvingKey: fixed / sigma column count does not match the constraint system")
        fa = (C.c_void_p * max(1, len(fx)))(*[c.ctypes.data for c in fx])
        sa = (C.c_void_p * max(1, len(sg)))(*[c.ctypes.data for c in sg])
        self._h = C.c_void_p()
        _check(lib().h2v_pk_load(params._h, C.byref(ct), fa, sa, _ptr(_fr1(vk_transcript_repr)), C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None) and self._h.value and _lib is not None:
            _lib.h2v_pk_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def proof_size(self):
        return int(lib().h2v_proof_size(self._h))

    def create_proof(self, advice, instances, rng_seed=bytes(32)):
        """`create_proof(params, pk, &[circuit], &[instances], ChaCha20Rng::from_seed(rng_seed), transcript)` -> proof bytes"""
        n = 1 << self.cs["k"]
        adv = [_fr(c, n) for c in advice]
        if len(adv) != self.cs["n_advice"] or len(instances) != self.cs["n_instance"]:
            raise ValueError("create_proof: advice / instance column count does not match the constraint system")
        inst = [_fr(np.asarray(c, dtype=np.uint64).reshape(-1, 4)) for c in instances]
        aa = (C.c_void_p * max(1, len(adv)))(*[c.ctypes.data for c in adv])
        ia = (C.c_void_p * max(1, len(inst)))(*[c.ctypes.data for c in inst])
        il = np.ascontiguousarray([c.shape[0] for c in inst] or [0], dtype=np.uint32)
        cap = self.proof_size()
        out = np.zeros(cap, dtype=np.uint8)
        ln = C.c_size_t()
        _check(lib().h2v_create_proof(self._h, aa, ia, _ptr(il), bytes(rng_seed), _ptr(out), cap, C.byref(ln)))
        return bytes(out[:ln.value])

    def create_proofs(self, advice_list, instances_list, rng_seeds):
        """Many proofs on this key in one call: proof p = create_proof(advice_list[p], instances_list[p], rng_seeds[p]),
        byte for byte.  The proofs run in groups, phase by phase (h2v_create_proofs) -> list of proof bytes"""
        B = len(advice_list)
        if len(instances_list) != B or len(rng_seeds) != B:
            raise ValueError("create_proofs: advice_list, instances_list and rng_seeds differ in length")
        if not B:
            return []
        n = 1 << self.cs["k"]
        keep, adv_ptrs, inst_ptrs, len_ptrs = [], [], [], []
        for p, (advice, instances, seed) in enumerate(zip(advice_list, instances_list, rng_seeds)):
            adv = [_fr(c, n) for c in advice]
            if len(adv) != self.cs["n_advice"] or len(instances) != self.cs["n_instance"]:
                raise ValueError(f"create_proofs: proof {p}: advice / instance column count does not match the constraint system")
            if len(bytes(seed)) != 32:
                raise ValueError(f"create_proofs: proof {p}: the rng seed is not 32 bytes")
            inst = [_fr(np.asarray(c, dtype=np.uint64).reshape(-1, 4)) for c in instances]
            aa = (C.c_void_p * max(1, len(adv)))(*[c.ctypes.data for c in adv])
            ia = (C.c_void_p * max(1, len(inst)))(*[c.ctypes.data for c in inst])
            il = np.ascontiguousarray([c.shape[0] for c in inst] or [0], dtype=np.uint32)
            keep += [adv, inst, aa, ia, il]
            adv_ptrs.append(C.cast(aa, C.c_void_p))
            inst_ptrs.append(C.cast(ia, C.c_void_p))
            len_ptrs.append(il.ctypes.data)
        seeds = b"".join(bytes(s_) for s_ in rng_seeds)
        size = self.proof_size()
        out = np.zeros(B * size, dtype=np.uint8)
        arr = lambda xs: (C.c_void_p * B)(*xs)
        _check(lib().h2v_create_proofs(self._h, B, arr(adv_ptrs), arr(inst_ptrs), arr(len_ptrs), seeds, _ptr(out), size))
        return [bytes(out[p * size:(p + 1) * size]) for p in range(B)]

    def mock_prover(self, advice_list, instances_list, max_failures=64):
        """MockProver.run on this key's circuit for every witness of a batch, in one call (h2v_pk_mock_prover): result w
        equals MockProver.run(cs, fixed, sigma, advice_list[w], instances_list[w], max_failures) with the key's cs, fixed
        and sigma.  Only the witnesses are uploaded; the key-only work is done by the first call -> list of MockProver"""
        B = len(advice_list)
        if len(instances_list) != B:
            raise ValueError("mock_prover: advice_list and instances_list differ in length")
        if not B:
            return []
        n = 1 << self.cs["k"]
        keep, adv_ptrs, inst_ptrs, len_ptrs = [], [], [], []
        for w, (advice, instances) in enumerate(zip(advice_list, instances_list)):
            adv = [_fr(c, n) for c in advice]
            if len(adv) != self.cs["n_advice"] or len(instances) != self.cs["n_instance"]:
                raise ValueError(f"mock_prover: witness {w}: advice / instance column count does not match the constraint system")
            inst = [_fr(np.asarray(c, dtype=np.uint64).reshape(-1, 4)) for c in instances]
            aa = (C.c_void_p * max(1, len(adv)))(*[c.ctypes.data for c in adv])
            ia = (C.c_void_p * max(1, len(inst)))(*[c.ctypes.data for c in inst])
            il = np.ascontiguousarray([c.shape[0] for c in inst] or [0], dtype=np.uint32)
            keep += [adv, inst, aa, ia, il]
            adv_ptrs.append(C.cast(aa, C.c_void_p))
            inst_ptrs.append(C.cast(ia, C.c_void_p))
            len_ptrs.append(il.ctypes.data)
        out = (_MockFailureT * max(1, B * max_failures))()
        totals = np.zeros(B, dtype=np.uint64)
        arr = lambda xs: (C.c_void_p * B)(*xs)
        _check(lib().h2v_pk_mock_prover(self._h, B, arr(adv_ptrs), arr(inst_ptrs), arr(len_ptrs), out, max_failures, _ptr(totals)))
        return _mock_results(B, out, totals, max_failures)

    def create_proofs_from_inputs(self, program, inputs_list, rng_seeds):
        """create_proofs on the columns program.generate(inputs_list) gives, byte for byte with the same seeds; the columns
        are generated in this key's device workspace and never reach the host (h2v_create_proofs_from_inputs).  The key
        must come from the recording's layout -> (proofs, instances), instances[p] as program.generate gives them"""
        B = len(inputs_list)
        if len(rng_seeds) != B:
            raise ValueError("create_proofs_from_inputs: inputs_list and rng_seeds differ in length")
        if not B:
            return [], []
        inp = program.pack_inputs(inputs_list, "create_proofs_from_inputs")
        if any(len(bytes(s_)) != 32 for s_ in rng_seeds):
            raise ValueError("create_proofs_from_inputs: an rng seed is not 32 bytes")
        seeds = b"".join(bytes(s_) for s_ in rng_seeds)
        size = self.proof_size()
        out = np.zeros(B * size, dtype=np.uint8)
        inst = np.zeros((B, program.info["instances"], 4), dtype=np.uint64)
        _check(lib().h2v_create_proofs_from_inputs(self._h, program._h, B, program.n_inputs, _ptr(inp), seeds, _ptr(out), size, _ptr(inst)))
        return [bytes(out[p * size:(p + 1) * size]) for p in range(B)], [[inst[p]] if self.cs["n_instance"] else [] for p in range(B)]

    def mock_prover_from_inputs(self, program, inputs_list, max_failures=64):
        """mock_prover on the columns program.generate(inputs_list) gives, generated in this key's device workspace
        (h2v_pk_mock_prover_from_inputs) -> list of MockProver (upload_ms: the generation)"""
        B = len(inputs_list)
        if not B:
            return []
        inp = program.pack_inputs(inputs_list, "mock_prover_from_inputs")
        out = (_MockFailureT * max(1, B * max_failures))()
        totals = np.zeros(B, dtype=np.uint64)
        _check(lib().h2v_pk_mock_prover_from_inputs(self._h, program._h, B, program.n_inputs, _ptr(inp), out, max_failures, _ptr(totals)))
        return _mock_results(B, out, totals, max_failures)

    def last_phase_ms(self):
        buf = (C.c_double * 8)()
        _check(lib().h2v_pk_last_phase_ms(self._h, buf))
        names = ["advice_commit", "lookup_permute", "grand_products", "transforms", "quotient", "evaluations", "multiopen"]
        return dict(zip(names, [float(x) for x in buf]))


# ----------------------------------------------------------------------------- dev/mock.rs MockProver
MOCK_GATE, MOCK_GATE_UNUSABLE, MOCK_LOOKUP, MOCK_SIGMA_NOT_DELTA_OMEGA, MOCK_SIGMA_NOT_PERMUTATION, MOCK_COPY_UNUSABLE, MOCK_COPY = range(1, 8)
MOCK_KINDS = {MOCK_GATE: "gate", MOCK_GATE_UNUSABLE: "gate_unusable", MOCK_LOOKUP: "lookup",
              MOCK_SIGMA_NOT_DELTA_OMEGA: "sigma_not_delta_omega", MOCK_SIGMA_NOT_PERMUTATION: "sigma_not_permutation",
              MOCK_COPY_UNUSABLE: "copy_unusable", MOCK_COPY: "copy"}
MockFailure = namedtuple("MockFailure", "kind column row other_column other_row")


class _MockFailureT(C.Structure):
    _fields_ = [(f, C.c_uint32) for f in MockFailure._fields]


def _mock_results(B, out, totals, max_failures):
    """the MockProver of each witness of the last h2v_pk_mock_prover* call"""
    ms = (C.c_double * 2)()
    _check(lib().h2v_mock_last_ms(ms))
    res = []
    for w in range(B):
        got = min(max_failures, int(totals[w]))
        fails = [MockFailure(*(getattr(out[w * max_failures + i], f) for f in MockFailure._fields)) for i in range(got)]
        res.append(MockProver(fails, int(totals[w]), ms[0], ms[1]))
    return res


class MockProver:
    """halo2 `MockProver::run(k, circuit, instances)` on the device (h2v_mock_prover): every gate, lookup and copy
    constraint of a laid-out circuit.  `failures`: the first max_failures failures (MockFailure, kind = MOCK_*) in the
    order gates, lookups, permutation; `n_failures`: how many there are in all; `upload_ms` / `check_ms`: the call's
    wall-clock time moving the columns to the device and checking them."""

    def __init__(self, failures, n_failures, upload_ms, check_ms):
        self.failures, self.n_failures, self.upload_ms, self.check_ms = failures, n_failures, upload_ms, check_ms

    @classmethod
    def run(cls, cs, fixed, sigma, advice, instances, max_failures=64):
        """cs as ProvingKey takes it; fixed / sigma / advice: Lagrange columns of 2^k Fr (Montgomery limbs, shape (n, 4));
        instances: one array of public inputs per instance column"""
        ct, _keep = _circuit_struct(cs)      # the index arrays ct points into
        n = 1 << cs["k"]
        fx, sg, adv = [_fr(c, n) for c in fixed], [_fr(c, n) for c in sigma], [_fr(c, n) for c in advice]
        inst = [_fr(np.asarray(c, dtype=np.uint64).reshape(-1, 4)) for c in instances]
        if (len(fx), len(sg), len(adv), len(inst)) != (cs["n_fixed"], len(cs["permutation"]), cs["n_advice"], cs["n_instance"]):
            raise ValueError("MockProver: fixed / sigma / advice / instance column count does not match the constraint system")
        arr = lambda cols: (C.c_void_p * max(1, len(cols)))(*[c.ctypes.data for c in cols])
        il = np.ascontiguousarray([c.shape[0] for c in inst] or [0], dtype=np.uint32)
        out = (_MockFailureT * max(1, max_failures))()
        total = C.c_uint64()
        _check(lib().h2v_mock_prover(C.byref(ct), arr(fx), arr(sg), arr(adv), arr(inst), _ptr(il), out, max_failures, C.byref(total)))
        ms = (C.c_double * 2)()
        _check(lib().h2v_mock_last_ms(ms))
        got = min(max_failures, total.value)
        fails = [MockFailure(*(getattr(out[i], f) for f in MockFailure._fields)) for i in range(got)]
        return cls(fails, total.value, ms[0], ms[1])

    def assert_satisfied(self):
        if self.n_failures:
            lines = [f"{MOCK_KINDS.get(f.kind, f.kind)}: column {f.column} row {f.row} (other: column {f.other_column} row {f.other_row})"
                     for f in self.failures[:16]]
            more = self.n_failures - len(lines)
            raise AssertionError(f"{self.n_failures} constraint(s) not satisfied:\n  " + "\n  ".join(lines)
                                 + (f"\n  ... and {more} more" if more > 0 else ""))


# ----------------------------------------------------------------------------- device self-tests
def selftest_field(field, op, a, b=None):
    a = np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, 4)
    out = np.zeros_like(a)
    bp = None
    if b is not None:
        b = np.ascontiguousarray(b, dtype=np.uint64).reshape(-1, 4)
        bp = _ptr(b)
    _check(lib().h2v_selftest_field(field, op, _ptr(a), bp, a.shape[0], _ptr(out)))
    return out


SYN_A, SYN_B = 0x9E3779B97F4A7C15 >> 2, 0x632BE59BD9B4E019 >> 2


def synthetic_bases(n, a=SYN_A, b=SYN_B):
    """bases[i] = (a*i + b) * G computed on the device (bench / full-size test inputs)."""
    out = np.zeros((n, 8), dtype=np.uint64)
    _check(lib().h2v_synthetic_bases(a, b, n, _ptr(out)))
    return out


def selftest_group(mode, p, q):
    p = np.ascontiguousarray(p, dtype=np.uint64).reshape(-1, 8)
    q = np.ascontiguousarray(q, dtype=np.uint64).reshape(-1, 8)
    out = np.zeros_like(p)
    _check(lib().h2v_selftest_group(mode, _ptr(p), _ptr(q), p.shape[0], _ptr(out)))
    return out
