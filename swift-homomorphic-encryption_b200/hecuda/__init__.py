"""hecuda -- host-side mirror of the reference's HeScheme surface for the RNS-BFV hot path, over libhecuda.so.

Names follow the reference (Sources/HomomorphicEncryption/HeScheme.swift): `Context`, `EvaluationKey`,
`Bfv.mulAssign / relinearize / modSwitchDown / forwardNtt / inverseNtt`.  Data crosses the boundary as numpy uint64
arrays shaped like the reference's Array2d-backed values:

    polynomial  : (rows, N)                  -- PolyRq.data            (PolyRq.swift:21-28)
    ciphertext  : (polys, rows, N)           -- Ciphertext.polys       (Ciphertext.swift:18-28)
    batch       : (batch, polys, rows, N)

Everything runs on the GPU through the C ABI in include/hecuda.h; there is no CPU fallback -- if the CUDA extension
is missing or no device is present, construction raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "libhecuda.so")

HECUDA_OK = 0
BASE_Q, BASE_Q_BSK, BASE_KEYSWITCH, BASE_Q_AUX = 0, 1, 2, 3
u64p = C.POINTER(C.c_uint64)

# every symbol include/hecuda.h declares: (restype, argtypes)
_VP = C.c_void_p
SYMBOLS = {
    "hecuda_version": (C.c_int32, []),
    "hecuda_last_error": (C.c_char_p, []),
    "hecuda_device_count": (C.c_int32, [C.POINTER(C.c_int32)]),
    "hecuda_set_device": (C.c_int32, [C.c_int32]),
    "hecuda_host_alloc": (C.c_int32, [C.POINTER(_VP), C.c_uint64]),
    "hecuda_host_free": (C.c_int32, [_VP]),
    "hecuda_host_register": (C.c_int32, [_VP, C.c_uint64]),
    "hecuda_host_unregister": (C.c_int32, [_VP]),
    "hecuda_context_create": (C.c_int32, [C.c_int64, u64p, C.c_int32, C.c_uint64, C.POINTER(_VP)]),
    "hecuda_context_destroy": (C.c_int32, [_VP]),
    "hecuda_context_ciphertext_moduli_count": (C.c_int32, [_VP, C.POINTER(C.c_int32)]),
    "hecuda_rnstool_lift_q_to_qbsk": (C.c_int32, [_VP, _VP, _VP, C.c_int64]),
    "hecuda_rnstool_floor_qbsk_to_q": (C.c_int32, [_VP, _VP, _VP, C.c_int64]),
    "hecuda_context_create_u32": (C.c_int32, [C.c_int64, _VP, C.c_int32, C.c_uint32, C.POINTER(_VP)]),
    "hecuda_context_word_bits": (C.c_int32, [_VP, C.POINTER(C.c_int32)]),
    "hecuda_u32_ntt_forward": (C.c_int32, [_VP, C.c_int32, _VP, C.c_int32, C.c_int64]),
    "hecuda_u32_ntt_inverse": (C.c_int32, [_VP, C.c_int32, _VP, C.c_int32, C.c_int64]),
    "hecuda_u32_bfv_multiply": (C.c_int32, [_VP, _VP, _VP, _VP, C.c_int64]),
    "hecuda_u32_evk_create": (C.c_int32, [_VP, _VP, C.POINTER(_VP)]),
    "hecuda_u32_bfv_relinearize": (C.c_int32, [_VP, _VP, _VP, C.c_int32, _VP, C.c_int64]),
    "hecuda_u32_bfv_mod_switch_down": (C.c_int32, [_VP, _VP, C.c_int32, C.c_int32, _VP, C.c_int64]),
    "hecuda_u32_bfv_multiply_relinearize": (C.c_int32, [_VP, _VP, _VP, _VP, C.c_int32, _VP, C.c_int64]),
    "hecuda_u32_bfv_relinearize_mod_switch_down": (C.c_int32, [_VP, _VP, _VP, C.c_int32, _VP, C.c_int64]),
    "hecuda_u32_evk_set_galois_key": (C.c_int32, [_VP, C.c_uint32, _VP]),
    "hecuda_u32_bfv_apply_galois": (C.c_int32, [_VP, _VP, _VP, C.c_int32, C.c_uint32, _VP, C.c_int64]),
    "hecuda_u32_bfv_inner_product": (C.c_int32, [_VP, _VP, _VP, _VP, C.c_int64, C.c_int64]),
    "hecuda_u32_rnstool_lift_q_to_qbsk": (C.c_int32, [_VP, _VP, _VP, C.c_int64]),
    "hecuda_u32_rnstool_floor_qbsk_to_q": (C.c_int32, [_VP, _VP, _VP, C.c_int64]),
    "hecuda_bfv_relinearize_mod_switch_down": (C.c_int32, [_VP, _VP, _VP, C.c_int32, _VP, C.c_int64]),
    "hecuda_bfv_multiply_relinearize": (C.c_int32, [_VP, _VP, _VP, _VP, C.c_int32, _VP, C.c_int64]),
    "hecuda_bfv_multiply_relinearize_device": (C.c_int32, [_VP, _VP, _VP, _VP, C.c_int32, _VP, C.c_int64, _VP]),
    "hecuda_comm_unique_id": (C.c_int32, [_VP]),
    "hecuda_comm_create": (C.c_int32, [_VP, C.c_int32, C.c_int32, C.POINTER(_VP)]),
    "hecuda_comm_destroy": (C.c_int32, [_VP]),
    "hecuda_evk_broadcast": (C.c_int32, [_VP, _VP, C.c_int32, C.c_int32, _VP, C.c_int32]),
    "hecuda_bind_host_to_device": (C.c_int32, [C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "hecuda_context_bsk_moduli": (C.c_int32, [_VP, u64p, C.c_int32, C.POINTER(C.c_int32)]),
    "hecuda_context_aux_moduli": (C.c_int32, [_VP, u64p, C.c_int32, C.POINTER(C.c_int32)]),
    "hecuda_context_root_tables": (C.c_int32, [_VP, C.c_uint64, u64p, u64p]),
    "hecuda_ntt_forward": (C.c_int32, [_VP, C.c_int32, _VP, C.c_int32, C.c_int64]),
    "hecuda_ntt_inverse": (C.c_int32, [_VP, C.c_int32, _VP, C.c_int32, C.c_int64]),
    "hecuda_ntt_forward_device": (C.c_int32, [_VP, C.c_int32, _VP, C.c_int32, C.c_int64, _VP]),
    "hecuda_ntt_inverse_device": (C.c_int32, [_VP, C.c_int32, _VP, C.c_int32, C.c_int64, _VP]),
    "hecuda_ntt_forward_rows": (C.c_int32, [_VP, C.c_uint64, _VP, C.c_int64]),
    "hecuda_ntt_inverse_rows": (C.c_int32, [_VP, C.c_uint64, _VP, C.c_int64]),
    "hecuda_bfv_multiply": (C.c_int32, [_VP, _VP, _VP, _VP, C.c_int64]),
    "hecuda_bfv_multiply_device": (C.c_int32, [_VP, _VP, _VP, _VP, C.c_int64, _VP]),
    "hecuda_evk_create": (C.c_int32, [_VP, _VP, C.POINTER(_VP)]),
    "hecuda_evk_destroy": (C.c_int32, [_VP]),
    "hecuda_evk_create_empty": (C.c_int32, [_VP, C.POINTER(_VP)]),
    "hecuda_evk_device_buffer": (C.c_int32, [_VP, C.POINTER(_VP), C.POINTER(C.c_uint64)]),
    "hecuda_bfv_relinearize": (C.c_int32, [_VP, _VP, _VP, C.c_int32, _VP, C.c_int64]),
    "hecuda_bfv_relinearize_device": (C.c_int32, [_VP, _VP, _VP, C.c_int32, _VP, C.c_int64, _VP]),
    "hecuda_bfv_mod_switch_down": (C.c_int32, [_VP, _VP, C.c_int32, C.c_int32, _VP, C.c_int64]),
    "hecuda_bfv_mod_switch_down_device": (C.c_int32, [_VP, _VP, C.c_int32, C.c_int32, _VP, C.c_int64, _VP]),
    "hecuda_evk_set_galois_key": (C.c_int32, [_VP, C.c_uint32, _VP]),
    "hecuda_evk_galois_device_buffer": (C.c_int32, [_VP, C.c_uint32, C.POINTER(_VP), C.POINTER(C.c_uint64)]),
    "hecuda_bfv_apply_galois": (C.c_int32, [_VP, _VP, _VP, C.c_int32, C.c_uint32, _VP, C.c_int64]),
    "hecuda_bfv_apply_galois_device": (C.c_int32, [_VP, _VP, _VP, C.c_int32, C.c_uint32, _VP, C.c_int64, _VP]),
    "hecuda_poly_apply_galois": (C.c_int32, [_VP, C.c_int32, C.c_int32, _VP, _VP, C.c_int32, C.c_int64, C.c_uint32]),
    "hecuda_bfv_inner_product_plaintexts": (C.c_int32, [_VP, _VP, C.c_int32, C.c_int32, C.c_int64, _VP, _VP, _VP, C.c_int64]),
    "hecuda_bfv_inner_product_plaintexts_device": (C.c_int32, [_VP, _VP, C.c_int32, C.c_int32, C.c_int64, _VP, _VP, _VP,
                                                                C.c_int64, _VP]),
    "hecuda_poly_multiply_power_of_x": (C.c_int32, [_VP, C.c_int32, _VP, _VP, C.c_int32, C.c_int64, C.c_int64]),
    "hecuda_bfv_inner_product": (C.c_int32, [_VP, _VP, _VP, _VP, C.c_int64, C.c_int64]),
    "hecuda_bfv_inner_product_device": (C.c_int32, [_VP, _VP, _VP, _VP, C.c_int64, C.c_int64, _VP]),
    "hecuda_plaintext_to_eval": (C.c_int32, [_VP, _VP, C.c_int32, _VP, C.c_int64]),
    "hecuda_plaintext_to_eval_device": (C.c_int32, [_VP, _VP, C.c_int32, _VP, C.c_int64, _VP]),
    "hecuda_pir_database_create": (C.c_int32, [_VP, _VP, C.c_int32, _VP, C.c_int64, C.POINTER(_VP)]),
    "hecuda_pir_database_destroy": (C.c_int32, [_VP]),
    "hecuda_pir_database_device_buffer": (C.c_int32, [_VP, C.POINTER(_VP), C.POINTER(C.c_uint64)]),
    "hecuda_mulpir_expand": (C.c_int32, [_VP, _VP, _VP, C.c_int32, C.c_int64, _VP]),
    "hecuda_mulpir_expand_device": (C.c_int32, [_VP, _VP, _VP, C.c_int32, C.c_int64, _VP, _VP]),
    "hecuda_mulpir_compute_response": (C.c_int32, [_VP, _VP, C.POINTER(_VP), C.c_int32, C.POINTER(C.c_int32), C.c_int32,
                                                   C.c_int32, _VP, C.c_int32, C.c_int32, _VP]),
    "hecuda_mulpir_compute_response_device": (C.c_int32, [_VP, _VP, C.POINTER(_VP), C.c_int32, C.POINTER(C.c_int32),
                                                          C.c_int32, C.c_int32, _VP, C.c_int32, C.c_int32, _VP, _VP]),
    "hecuda_mulpir_compute_response_wire": (C.c_int32, [_VP, _VP, C.POINTER(_VP), C.c_int32, C.POINTER(C.c_int32), C.c_int32,
                                                        C.c_int32, _VP, _VP, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _VP]),
    "hecuda_pnns_matrix_create": (C.c_int32, [_VP, _VP, C.c_int32, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.POINTER(_VP)]),
    "hecuda_pnns_matrix_destroy": (C.c_int32, [_VP]),
    "hecuda_pnns_matrix_result_count": (C.c_int32, [_VP, C.POINTER(C.c_int64)]),
    "hecuda_pnns_mul_transpose_vector": (C.c_int32, [_VP, _VP, _VP, _VP, C.c_int64, C.c_int32, _VP]),
    "hecuda_pnns_mul_transpose_vector_device": (C.c_int32, [_VP, _VP, _VP, _VP, C.c_int64, C.c_int32, _VP, _VP]),
    "hecuda_pnns_mul_transpose_matrix": (C.c_int32, [_VP, _VP, _VP, _VP, C.c_int32, C.c_int32, C.POINTER(C.c_int32), _VP,
                                                     C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.c_int32,
                                                     _VP, C.c_int64, C.POINTER(C.c_int64)]),
    "hecuda_poly_serialized_byte_count": (C.c_int32, [_VP, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_uint64)]),
    "hecuda_poly_serialize": (C.c_int32, [_VP, C.c_int32, _VP, C.c_int32, _VP, C.c_int32, C.c_int64]),
    "hecuda_poly_load": (C.c_int32, [_VP, C.c_int32, _VP, C.c_int32, _VP, C.c_int32, C.c_int64]),
    "hecuda_poly_serialize_device": (C.c_int32, [_VP, C.c_int32, _VP, C.c_int32, _VP, C.c_int32, C.c_int64, _VP]),
    "hecuda_poly_load_device": (C.c_int32, [_VP, C.c_int32, _VP, C.c_int32, _VP, C.c_int32, C.c_int64, _VP]),
    "hecuda_poly_random_from_seed": (C.c_int32, [_VP, _VP, C.c_int32, _VP, C.c_int64]),
    "hecuda_ciphertext_expand_seeded": (C.c_int32, [_VP, _VP, _VP, C.c_int32, _VP, C.c_int64]),
    "hecuda_bfv_decrypt": (C.c_int32, [_VP, _VP, _VP, C.c_int32, C.c_int32, C.c_uint64, _VP, C.c_int64]),
    "hecuda_poly_add": (C.c_int32, [_VP, C.c_int32, _VP, _VP, C.c_int32, C.c_int64]),
    "hecuda_poly_add_device": (C.c_int32, [_VP, C.c_int32, _VP, _VP, C.c_int32, C.c_int64, _VP]),
    "hecuda_poly_sub": (C.c_int32, [_VP, C.c_int32, _VP, _VP, C.c_int32, C.c_int64]),
    "hecuda_poly_sub_device": (C.c_int32, [_VP, C.c_int32, _VP, _VP, C.c_int32, C.c_int64, _VP]),
    "hecuda_poly_mul": (C.c_int32, [_VP, C.c_int32, _VP, _VP, C.c_int32, C.c_int64]),
    "hecuda_poly_mul_device": (C.c_int32, [_VP, C.c_int32, _VP, _VP, C.c_int32, C.c_int64, _VP]),
    "hecuda_poly_neg": (C.c_int32, [_VP, C.c_int32, _VP, C.c_int32, C.c_int64]),
    "hecuda_poly_neg_device": (C.c_int32, [_VP, C.c_int32, _VP, C.c_int32, C.c_int64, _VP]),
    "hecuda_poly_mul_scalars": (C.c_int32, [_VP, C.c_int32, _VP, _VP, C.c_int32, C.c_int64]),
    "hecuda_poly_mul_scalars_device": (C.c_int32, [_VP, C.c_int32, _VP, _VP, C.c_int32, C.c_int64, _VP]),
    "hecuda_kernel_launch_count": (C.c_uint64, []),
}

_lib = None


class HeError(RuntimeError):
    """Mirrors `throws HeError` (Sources/HomomorphicEncryption/Error.swift:17-54)."""

    def __init__(self, code: int, message: str):
        super().__init__(f"[{code}] {message}")
        self.code = code
        self.message = message


def load_library(path: str = LIB_PATH):
    """dlopen libhecuda.so and bind every declared symbol.  Raises if the library or a symbol is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(path):
            raise HeError(-4, f"libhecuda.so not found at {path}: build it with __graft_entry__.build() "
                              "(the product has no CPU fallback)")
        lib = C.CDLL(path)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)  # AttributeError if the .so does not export it
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def _check(rc: int):
    if rc != HECUDA_OK:
        raise HeError(rc, (load_library().hecuda_last_error() or b"").decode())


def _host(a, dtype=np.uint64) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a, dtype=dtype))


def _ptr(a: np.ndarray):
    return C.c_void_p(a.ctypes.data)


def device_count() -> int:
    n = C.c_int32(0)
    rc = load_library().hecuda_device_count(C.byref(n))
    return n.value if rc == HECUDA_OK else 0


def set_device(i: int):
    _check(load_library().hecuda_set_device(i))


class Communicator:
    """NCCL communicator of the evaluation-key broadcast, through the C ABI (hecuda_comm_*): what a torch-free host uses.
    Rank 0 calls Communicator.uniqueId() and hands the 128 bytes to the other ranks; every rank then constructs the
    communicator (collective) and calls broadcast (collective) on its EvaluationKey."""

    @staticmethod
    def uniqueId() -> bytes:
        buf = (C.c_uint8 * 128)()
        _check(load_library().hecuda_comm_unique_id(buf))
        return bytes(buf)

    def __init__(self, unique_id: bytes, rank: int, world_size: int):
        h = C.c_void_p()
        buf = (C.c_uint8 * 128).from_buffer_copy(unique_id)
        _check(load_library().hecuda_comm_create(buf, rank, world_size, C.byref(h)))
        self._h, self.rank, self.world_size = h, rank, world_size

    def broadcast(self, key: "EvaluationKey", root: int = 0, has_relin: bool = True, galois_elements=()):
        elems = (C.c_uint32 * max(1, len(galois_elements)))(*[int(e) for e in galois_elements])
        _check(load_library().hecuda_evk_broadcast(key._h, self._h, root, 1 if has_relin else 0, elems, len(galois_elements)))
        return key

    def close(self):
        if self._h is not None:
            load_library().hecuda_comm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def bind_host_to_device(device: int) -> dict:
    """Pins this thread (and threads created later) to the CPUs next to GPU `device` and prefers its NUMA node for
    page allocations (hecuda_bind_host_to_device).  Call once per process after set_device, before allocating
    PinnedBuffers.  Returns {"numa_node": n, "cpus": count} (numa_node -1 = not reported, nothing changed)."""
    node, cpus = C.c_int32(-1), C.c_int32(0)
    _check(load_library().hecuda_bind_host_to_device(device, C.byref(node), C.byref(cpus)))
    return {"numa_node": node.value, "cpus": cpus.value}


def kernel_launch_count() -> int:
    return int(load_library().hecuda_kernel_launch_count())


class PinnedBuffer:
    """Page-locked host array (hecuda_host_alloc) so the host-pointer entry points can overlap their copies."""

    def __init__(self, shape, dtype=np.uint64):
        self.nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = C.c_void_p()
        _check(load_library().hecuda_host_alloc(C.byref(p), max(self.nbytes, 8)))
        self._p = p
        buf = (C.c_char * max(self.nbytes, 8)).from_address(p.value)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def free(self):
        if self._p is not None:
            self.array = None
            load_library().hecuda_host_free(self._p)
            self._p = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Context:
    """Context<Bfv<T>> (Context.swift:19,94-143).  coefficient_moduli = [q_0 .. q_{L-1}, q_ks].
    scalar = np.uint64 (default) is Context<Bfv<UInt64>>; np.uint32 is Context<Bfv<UInt32>> (use the Bfv32 operations)."""

    def __init__(self, poly_degree: int, coefficient_moduli, plaintext_modulus: int, scalar=np.uint64):
        lib = load_library()
        self.degree = int(poly_degree)
        self.coefficientModuli = [int(m) for m in coefficient_moduli]
        self.plaintextModulus = int(plaintext_modulus)
        self.scalar = np.dtype(scalar)
        h = C.c_void_p()
        if self.scalar == np.dtype(np.uint32):
            mods = np.ascontiguousarray(self.coefficientModuli, dtype=np.uint64)
            if mods.size and int(mods.max()) >> 32:
                raise HeError(-1, "invalidModulus: coefficient modulus does not fit UInt32")
            mods = mods.astype(np.uint32)
            _check(lib.hecuda_context_create_u32(self.degree, _ptr(mods), len(mods), self.plaintextModulus, C.byref(h)))
        else:
            mods = _host(self.coefficientModuli)
            _check(lib.hecuda_context_create(self.degree, mods.ctypes.data_as(u64p), len(mods), self.plaintextModulus,
                                             C.byref(h)))
        self._h = h
        n = C.c_int32(0)
        _check(lib.hecuda_context_ciphertext_moduli_count(h, C.byref(n)))
        self.L = n.value
        out = np.zeros(self.L + 1, dtype=np.uint64)
        _check(lib.hecuda_context_bsk_moduli(h, out.ctypes.data_as(u64p), len(out), C.byref(n)))
        self.bskModuli = [int(v) for v in out]
        _check(lib.hecuda_context_aux_moduli(h, out.ctypes.data_as(u64p), len(out), C.byref(n)))
        self.auxModuli = [int(v) for v in out]  # the base Bfv.mulAssign computes in (BASE_Q_AUX)

    @property
    def ciphertextModuli(self):
        return self.coefficientModuli[: self.L]

    def close(self):
        if getattr(self, "_h", None) is not None:
            load_library().hecuda_context_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def rootTables(self, modulus: int):
        roots = np.zeros(self.degree, dtype=np.uint64)
        inv = np.zeros(self.degree, dtype=np.uint64)
        _check(load_library().hecuda_context_root_tables(self._h, modulus, roots.ctypes.data_as(u64p),
                                                         inv.ctypes.data_as(u64p)))
        return roots, inv


class EvaluationKey:
    """EvaluationKey<Bfv<UInt64>> holding the relinearization key (Keys.swift:66-99,222)."""

    _dtype, _prefix = np.uint64, "hecuda_"  # key words and entry points of this width

    def __init__(self, context: Context, relinearizationKey=None):
        self.context = context
        self.galoisElements = []  # EvaluationKey.config.galoisElements
        h = C.c_void_p()
        if relinearizationKey is None:
            _check(load_library().hecuda_evk_create_empty(context._h, C.byref(h)))
        else:
            key = self._key(relinearizationKey, "relinearization")
            _check(getattr(load_library(), self._prefix + "evk_create")(context._h, _ptr(key), C.byref(h)))
        self._h = h

    def _key(self, key, kind: str) -> np.ndarray:
        k = _host(key, self._dtype)
        if k.size != self.context.L * 2 * (self.context.L + 1) * self.context.degree:
            raise HeError(-1, f"invalidContext: {kind} key must be L x 2 x (L+1) x N")
        return k

    def setGaloisKey(self, element: int, key):
        """GaloisKey.keys[element] (Keys.swift:150-163): (L, 2, L+1, N), Eval format."""
        k = self._key(key, "Galois")
        _check(getattr(load_library(), self._prefix + "evk_set_galois_key")(self._h, int(element), _ptr(k)))
        if element not in self.galoisElements:
            self.galoisElements.append(int(element))

    def deviceBuffer(self):
        p, n = C.c_void_p(), C.c_uint64(0)
        _check(load_library().hecuda_evk_device_buffer(self._h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def galoisDeviceBuffer(self, element: int):
        """Device buffer of GaloisKey.keys[element], allocated if absent (filled by a collective on non-source ranks)."""
        p, n = C.c_void_p(), C.c_uint64(0)
        _check(load_library().hecuda_evk_galois_device_buffer(self._h, element, C.byref(p), C.byref(n)))
        if element not in self.galoisElements:
            self.galoisElements.append(int(element))
        return p.value, n.value

    def close(self):
        if getattr(self, "_h", None) is not None:
            load_library().hecuda_evk_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class EvaluationKey32(EvaluationKey):
    """EvaluationKey<Bfv<UInt32>>: the keys as uint32 (L x 2 x (L+1) x N, Eval)."""

    _dtype, _prefix = np.uint32, "hecuda_u32_"

    def __init__(self, context: Context, relin_key):
        super().__init__(context, relin_key)


class _BfvOps:
    """The Bfv methods that have a uint64 (hecuda_*) and a uint32 (hecuda_u32_*) entry point, written once: Bfv binds
    them to uint64 arrays, Bfv32 to uint32 arrays.  The array shapes are checked here, before the library reads or
    writes them."""

    _dtype, _prefix = np.uint64, "hecuda_"

    @classmethod
    def _call(cls, name: str, *args):
        _check(getattr(load_library(), cls._prefix + name)(*args))

    @classmethod
    def _out(cls, out, shape):
        return np.empty(shape, dtype=cls._dtype) if out is None else out

    @classmethod
    def mulAssign(cls, context: Context, lhs, rhs, out=None):
        """Bfv.mulAssign (Bfv+Multiply.swift:18-21): (batch, 2, L, N) x (batch, 2, L, N) -> (batch, 3, L, N)."""
        a, b = _host(lhs, cls._dtype), _host(rhs, cls._dtype)
        shape = (2, context.L, context.degree)
        if a.shape[-3:] != shape or b.shape != a.shape:
            raise HeError(-1, f"invalidCiphertext: expected (..., 2, {context.L}, {context.degree}), got {a.shape} and {b.shape}")
        batch = int(np.prod(a.shape[:-3], dtype=np.int64))
        out = cls._out(out, a.shape[:-3] + (3, context.L, context.degree))
        cls._call("bfv_multiply", context._h, _ptr(a), _ptr(b), _ptr(out), batch)
        return out

    @classmethod
    def relinearizeModSwitchDown(cls, context: Context, ciphertext, key: EvaluationKey, out=None):
        """relinearize + modSwitchDown in one pass (hecuda_bfv_relinearize_mod_switch_down): (batch, 3, l, N) -> (batch, 2, l-1, N)."""
        c = _host(ciphertext, cls._dtype)
        if c.ndim < 3 or c.shape[-3] != 3 or c.shape[-1] != context.degree:
            raise HeError(-1, "invalidCiphertext: ciphertext must have three polys when relinearizing")
        if key is None:
            raise HeError(-5, "missingRelinearizationKey")
        l = c.shape[-2]
        batch = int(np.prod(c.shape[:-3], dtype=np.int64))
        out = cls._out(out, c.shape[:-3] + (2, l - 1, context.degree))
        cls._call("bfv_relinearize_mod_switch_down", context._h, key._h, _ptr(c), l, _ptr(out), batch)
        return out

    @classmethod
    def mulRelinearize(cls, context: Context, lhs, rhs, key: EvaluationKey, modSwitchDown: bool = False, out=None):
        """mulAssign + relinearize (+ modSwitchDown) in one pass (hecuda_bfv_multiply_relinearize): (batch, 2, L, N) x2 ->
        (batch, 2, L, N) or (batch, 2, L-1, N).  Same residues as the separate calls."""
        a, b = _host(lhs, cls._dtype), _host(rhs, cls._dtype)
        L, n = context.L, context.degree
        if a.shape != b.shape or a.shape[-3:] != (2, L, n):
            raise HeError(-1, "invalidCiphertext: multiply takes top-level two-polynomial ciphertexts")
        if key is None:
            raise HeError(-5, "missingRelinearizationKey")
        rows = L - 1 if modSwitchDown else L
        out = cls._out(out, a.shape[:-3] + (2, rows, n))
        cls._call("bfv_multiply_relinearize", context._h, key._h, _ptr(a), _ptr(b), 1 if modSwitchDown else 0, _ptr(out),
                  a.size // (2 * L * n))
        return out

    @classmethod
    def relinearize(cls, context: Context, ciphertext, key: EvaluationKey, out=None):
        """Bfv.relinearize (Bfv.swift:201-219): (batch, 3, l, N) -> (batch, 2, l, N)."""
        c = _host(ciphertext, cls._dtype)
        if c.ndim < 3 or c.shape[-3] != 3 or c.shape[-1] != context.degree:
            raise HeError(-1, "invalidCiphertext: ciphertext must have three polys when relinearizing")
        if key is None:
            raise HeError(-5, "missingRelinearizationKey")
        l = c.shape[-2]
        batch = int(np.prod(c.shape[:-3], dtype=np.int64))
        out = cls._out(out, c.shape[:-3] + (2, l, context.degree))
        cls._call("bfv_relinearize", context._h, key._h, _ptr(c), l, _ptr(out), batch)
        return out

    @classmethod
    def modSwitchDown(cls, context: Context, ciphertext, out=None):
        """Bfv.modSwitchDown (Bfv.swift:163-171): (batch, polys, l, N) -> (batch, polys, l-1, N)."""
        c = _host(ciphertext, cls._dtype)
        if c.ndim < 3 or c.shape[-1] != context.degree:
            raise HeError(-1, "invalidCiphertext")
        polys, l = c.shape[-3], c.shape[-2]
        batch = int(np.prod(c.shape[:-3], dtype=np.int64))
        out = cls._out(out, c.shape[:-3] + (polys, l - 1, context.degree))
        cls._call("bfv_mod_switch_down", context._h, _ptr(c), polys, l, _ptr(out), batch)
        return out

    @classmethod
    def applyGalois(cls, context: Context, ciphertext, element: int, key: EvaluationKey, out=None):
        """Bfv.applyGalois (Bfv.swift:174-198): (batch, 2, l, N) -> (batch, 2, l, N)."""
        c = _host(ciphertext, cls._dtype)
        if c.ndim < 3 or c.shape[-3] != 2 or c.shape[-1] != context.degree:
            raise HeError(-1, "invalidCiphertext: ciphertext must have two polys when applying galois")
        if key is None:
            raise HeError(-5, "missingGaloisKey")
        l = c.shape[-2]
        batch = int(np.prod(c.shape[:-3], dtype=np.int64))
        out = cls._out(out, c.shape)
        cls._call("bfv_apply_galois", context._h, key._h, _ptr(c), l, int(element), _ptr(out), batch)
        return out

    @classmethod
    def innerProductCiphertexts(cls, context: Context, lhs, rhs):
        """Bfv.innerProduct(_:_:) (Bfv.swift:315-361): (groups, pairs, 2, L, N) x same -> (groups, 3, L, N)."""
        a, b = _host(lhs, cls._dtype), _host(rhs, cls._dtype)
        if a.ndim != 5 or a.shape != b.shape or a.shape[2:] != (2, context.L, context.degree):
            raise HeError(-1, f"invalidCiphertext: expected (groups, pairs, 2, {context.L}, {context.degree})")
        out = np.empty((a.shape[0], 3, context.L, context.degree), dtype=cls._dtype)
        cls._call("bfv_inner_product", context._h, _ptr(a), _ptr(b), _ptr(out), a.shape[1], a.shape[0])
        return out

    @classmethod
    def liftQToQBsk(cls, context: Context, polys):
        """_RnsTool.liftQToQBsk (RnsTool.swift:324-331): (..., L, N) Coeff -> (..., 2L+1, N) over [Q, Bsk]."""
        d = _host(polys, cls._dtype)
        L, n = context.L, context.degree
        if d.shape[-2:] != (L, n):
            raise HeError(-1, "invalidPolyContext: liftQToQBsk takes top-level polynomials")
        out = np.empty(d.shape[:-2] + (2 * L + 1, n), dtype=cls._dtype)
        cls._call("rnstool_lift_q_to_qbsk", context._h, _ptr(d), _ptr(out), d.size // (L * n))
        return out

    @classmethod
    def floorQBskToQ(cls, context: Context, polys):
        """_RnsTool.floorQBskToQ (RnsTool.swift:453-456): (..., 2L+1, N) Coeff over [Q, Bsk] -> (..., L, N)."""
        d = _host(polys, cls._dtype)
        L, n = context.L, context.degree
        if d.shape[-2:] != (2 * L + 1, n):
            raise HeError(-1, "invalidPolyContext: floorQBskToQ takes polynomials over [Q, Bsk]")
        out = np.empty(d.shape[:-2] + (L, n), dtype=cls._dtype)
        cls._call("rnstool_floor_qbsk_to_q", context._h, _ptr(d), _ptr(out), d.size // ((2 * L + 1) * n))
        return out

    @classmethod
    def _ntt(cls, name: str, context: Context, polys, base: int):
        d = _host(polys, cls._dtype).copy()
        if d.ndim < 2 or d.shape[-1] != context.degree:
            raise HeError(-1, f"invalidPolyContext: expected (..., rows, {context.degree}), got {d.shape}")
        rows = d.shape[-2]
        cls._call(name, context._h, base, _ptr(d), rows, d.size // (rows * context.degree))
        return d

    @classmethod
    def forwardNtt(cls, context: Context, polys, base: int = BASE_Q):
        """PolyRq.forwardNtt (PolyRq+Ntt.swift:230): (..., rows, N) Coeff -> Eval."""
        return cls._ntt("ntt_forward", context, polys, base)

    @classmethod
    def inverseNtt(cls, context: Context, polys, base: int = BASE_Q):
        """PolyRq.inverseNtt (PolyRq+Ntt.swift:541): (..., rows, N) Eval -> Coeff."""
        return cls._ntt("ntt_inverse", context, polys, base)


class Bfv(_BfvOps):
    """enum Bfv<UInt64>: HeScheme -- the hot-path statics (Bfv/Bfv.swift:20), batched over a leading axis."""

    @staticmethod
    def polyApplyGalois(context: Context, polys, element: int, evalFormat: bool = False, base: int = BASE_Q):
        """PolyRq.applyGalois(element:) (Galois.swift:115-141 Coeff, :151-166 Eval) on (..., rows, N)."""
        d = _host(polys)
        rows = d.shape[-2]
        out = np.empty_like(d)
        _check(load_library().hecuda_poly_apply_galois(context._h, base, int(evalFormat), _ptr(d), _ptr(out), rows,
                                                       d.size // (rows * context.degree), element))
        return out

    @staticmethod
    def innerProduct(context: Context, ciphertexts, plaintexts, present=None):
        """Bfv.innerProduct(ciphertexts:plaintexts:) (Bfv.swift:476-505), batched over plaintext rows:
        ciphertexts (terms, polys, l, N) Eval; plaintexts (rows, terms, l, N) Eval; present (rows, terms) flags
        (False = nil plaintext) -> (rows, polys, l, N) Eval."""
        c, p = _host(ciphertexts), _host(plaintexts)
        if c.ndim != 4 or c.shape[-1] != context.degree:
            raise HeError(-1, "invalidCiphertext: expected (terms, polys, l, N)")
        terms, polys, l = c.shape[0], c.shape[1], c.shape[2]
        p = p.reshape(-1, terms, l, context.degree)
        out = np.empty((p.shape[0], polys, l, context.degree), dtype=np.uint64)
        pres = None
        if present is not None:
            pres = np.ascontiguousarray(np.asarray(present, dtype=np.uint8)).reshape(p.shape[0], terms)
        _check(load_library().hecuda_bfv_inner_product_plaintexts(
            context._h, _ptr(c), polys, l, terms, _ptr(p), C.c_void_p(pres.ctypes.data) if pres is not None else None,
            _ptr(out), p.shape[0]))
        return out

    @staticmethod
    def multiplyPowerOfX(context: Context, polys, power: int, base: int = BASE_Q):
        """PolyRq.multiplyPowerOfX (PolyRq.swift:398-422) on (..., rows, N) Coeff polynomials."""
        d = _host(polys)
        rows = d.shape[-2]
        out = np.empty_like(d)
        _check(load_library().hecuda_poly_multiply_power_of_x(context._h, base, _ptr(d), _ptr(out), rows,
                                                              d.size // (rows * context.degree), power))
        return out

    @staticmethod
    def plaintextToEval(context: Context, plaintexts, moduliCount: int = 0):
        """Plaintext.convertToEvalFormat (Plaintext.swift:149-171): (count, N) values < t -> (count, l, N) Eval."""
        d = _host(plaintexts).reshape(-1, context.degree)
        l = moduliCount or context.L
        out = np.empty((d.shape[0], l, context.degree), dtype=np.uint64)
        _check(load_library().hecuda_plaintext_to_eval(context._h, _ptr(d), l, _ptr(out), d.shape[0]))
        return out

    @staticmethod
    def randomPolys(context: Context, seeds, moduliCount: int = 0) -> np.ndarray:
        """PolyRq.random(context:using: NistAes128Ctr(seed:)) for (batch, 32) uint8 seeds -> (batch, l, N)."""
        sd = np.ascontiguousarray(np.asarray(seeds, dtype=np.uint8)).reshape(-1, 32)
        l = moduliCount or context.L
        out = np.empty((sd.shape[0], l, context.degree), dtype=np.uint64)
        _check(load_library().hecuda_poly_random_from_seed(context._h, sd.ctypes.data_as(C.c_void_p), l, _ptr(out), sd.shape[0]))
        return out

    @staticmethod
    def expandSeeded(context: Context, poly0, seeds, moduliCount: int = 0) -> np.ndarray:
        """Ciphertext(deserialize: .seeded(poly0:seed:)) (SerializedCiphertext.swift:41-60) -> (batch, 2, l, N) Coeff."""
        sd = np.ascontiguousarray(np.asarray(seeds, dtype=np.uint8)).reshape(-1, 32)
        l = moduliCount or context.L
        size = Bfv.serializationByteCount(context, l)
        p0 = np.ascontiguousarray(np.asarray(poly0, dtype=np.uint8)).reshape(-1)
        if p0.size != size * sd.shape[0]:
            raise HeError(-1, f"serializedBufferSizeMismatch(actual: {p0.size}, expected: {size * sd.shape[0]})")
        out = np.empty((sd.shape[0], 2, l, context.degree), dtype=np.uint64)
        _check(load_library().hecuda_ciphertext_expand_seeded(context._h, p0.ctypes.data_as(C.c_void_p),
                                                              sd.ctypes.data_as(C.c_void_p), l, _ptr(out), sd.shape[0]))
        return out

    @staticmethod
    def _elementwise(name: str, context: Context, lhs, rhs, base: int):
        a = _host(lhs).copy()
        rows = a.shape[-2]
        count = a.size // (rows * context.degree)
        fn = getattr(load_library(), "hecuda_poly_" + name)
        if rhs is None:
            _check(fn(context._h, base, _ptr(a), rows, count))
        else:
            b = _host(rhs)
            if name != "mul_scalars" and b.shape != a.shape:
                raise HeError(-1, "invalidPolyContext: operand shapes differ")
            _check(fn(context._h, base, _ptr(a), _ptr(b), rows, count))
        return a

    @staticmethod
    def polyAdd(context: Context, lhs, rhs, base: int = BASE_Q):
        """PolyRq + PolyRq (PolyRq.swift:147-157) on (..., rows, N) arrays."""
        return Bfv._elementwise("add", context, lhs, rhs, base)

    @staticmethod
    def polySub(context: Context, lhs, rhs, base: int = BASE_Q):
        return Bfv._elementwise("sub", context, lhs, rhs, base)

    @staticmethod
    def polyMul(context: Context, lhs, rhs, base: int = BASE_Q):
        """PolyRq<Eval> * PolyRq<Eval> (PolyRq.swift:184-204)."""
        return Bfv._elementwise("mul", context, lhs, rhs, base)

    @staticmethod
    def polyNeg(context: Context, poly, base: int = BASE_Q):
        return Bfv._elementwise("neg", context, poly, None, base)

    @staticmethod
    def polyMulScalars(context: Context, poly, scalars, base: int = BASE_Q):
        """PolyRq *= [T] (PolyRq.swift:232-245): one reduced scalar per RNS row."""
        return Bfv._elementwise("mul_scalars", context, poly, np.asarray(scalars, dtype=np.uint64), base)

    @staticmethod
    def decrypt(context: Context, ciphertexts, secretKey, scalingFactor: int = 1) -> np.ndarray:
        """Bfv.decryptCoeff (Bfv+Decrypt.swift:21-41): (batch, polys, l, N) Coeff ciphertexts -> (batch, N) coefficients < t.
        secretKey: SecretKey.poly, (L+1, N) in Eval format."""
        cts = _host(ciphertexts)
        if cts.ndim == 3:
            cts = cts[None]
        batch, polys, l, n = cts.shape
        sk = _host(secretKey)
        if sk.size < l * n:
            raise HeError(-1, "invalidContext: secret key has too few rows")
        out = np.empty((batch, n), dtype=np.uint64)
        _check(load_library().hecuda_bfv_decrypt(context._h, _ptr(sk), _ptr(cts), polys, l, scalingFactor, _ptr(out), batch))
        return out

    @staticmethod
    def serializationByteCount(context: Context, rowCount: int, skipLSBs: int = 0, base: int = BASE_Q) -> int:
        """PolyContext.serializationByteCount(skipLSBs:) (PolyRq+Serialize.swift:86-96)."""
        n = C.c_uint64(0)
        _check(load_library().hecuda_poly_serialized_byte_count(context._h, base, rowCount, skipLSBs, C.byref(n)))
        return n.value

    @staticmethod
    def serialize(context: Context, polys, skipLSBs: int = 0, base: int = BASE_Q) -> np.ndarray:
        """PolyRq.serialize(skipLSBs:) for polys of shape (..., rows, N) -> uint8 array (count, byteCount)."""
        x = _host(polys)
        rows = x.shape[-2]
        count = x.size // (rows * context.degree)
        size = Bfv.serializationByteCount(context, rows, skipLSBs, base)
        out = np.empty((count, size), dtype=np.uint8)
        _check(load_library().hecuda_poly_serialize(context._h, base, _ptr(x), skipLSBs, out.ctypes.data_as(C.c_void_p), rows, count))
        return out

    @staticmethod
    def load(context: Context, serialized, rowCount: int, skipLSBs: int = 0, base: int = BASE_Q) -> np.ndarray:
        """PolyRq.load(from:skipLSBs:): uint8 (count, byteCount) -> (count, rows, N) uint64."""
        b = np.ascontiguousarray(np.asarray(serialized, dtype=np.uint8))
        size = Bfv.serializationByteCount(context, rowCount, skipLSBs, base)
        if b.size % size:
            raise HeError(-1, f"serializedBufferSizeMismatch(actual: {b.size}, expected: a multiple of {size})")
        count = b.size // size
        out = np.empty((count, rowCount, context.degree), dtype=np.uint64)
        _check(load_library().hecuda_poly_load(context._h, base, b.ctypes.data_as(C.c_void_p), skipLSBs, _ptr(out), rowCount, count))
        return out

    @staticmethod
    def forwardNttRows(context: Context, modulus: int, rows):
        """PolyContext.forwardNtt(dataPtr:modulus:) (PolyRq+Ntt.swift:329-347)."""
        d = _host(rows).copy()
        _check(load_library().hecuda_ntt_forward_rows(context._h, modulus, _ptr(d), d.size // context.degree))
        return d

    @staticmethod
    def inverseNttRows(context: Context, modulus: int, rows):
        d = _host(rows).copy()
        _check(load_library().hecuda_ntt_inverse_rows(context._h, modulus, _ptr(d), d.size // context.degree))
        return d


class Bfv32(_BfvOps):
    """The Bfv<UInt32> data path (uint32 arrays, Context(..., scalar=np.uint32)): same shapes as the Bfv methods."""

    _dtype, _prefix = np.uint32, "hecuda_u32_"
