"""ctypes binding of libb2m.so (include/b2m.h).  No fallback: if the CUDA library is missing
or fails to load, importing the product raises."""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb2m.so")

CURVE_BLS12_381 = 0
CURVE_BN254 = 1
PC_MARLIN_KZG10 = 0
PC_SONIC_KZG10 = 1
RNG_CHACHA8, RNG_CHACHA12, RNG_CHACHA20 = 8, 12, 20
VERDICT_ACCEPT, VERDICT_REJECT, VERDICT_MALFORMED = 0, 1, 2

# (Fr u64 limbs, Fq u64 limbs) per curve id
LIMBS = {CURVE_BLS12_381: (4, 6), CURVE_BN254: (4, 4)}


class B2MError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"b2m error {code}: {msg}")
        self.code = code


class Matrix(ctypes.Structure):
    _fields_ = [("row_ptr", ctypes.c_void_p), ("col", ctypes.c_void_p), ("coeff", ctypes.c_void_p)]


NEXT_U64 = ctypes.CFUNCTYPE(ctypes.c_uint64, ctypes.c_void_p)
RNG_CALLBACK = 1


class Rng(ctypes.Structure):
    _fields_ = [("kind", ctypes.c_int), ("key", ctypes.c_uint8 * 32), ("word_pos", ctypes.c_uint64), ("next_u64", NEXT_U64),
                ("state", ctypes.c_void_p)]


_lib = None


def lib():
    """Load libb2m.so once.  Fails loudly when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not found: build it with `make -C marlin_b200/csrc -j8` "
                "(or __graft_entry__.build()); marlin_b200 has no CPU fallback")
        L = ctypes.CDLL(LIB_PATH)
        vp, cp, u64, sz, ci = ctypes.c_void_p, ctypes.c_char_p, ctypes.c_uint64, ctypes.c_size_t, ctypes.c_int
        P = ctypes.POINTER
        L.b2m_last_error.restype = cp
        L.b2m_version.restype = cp
        L.b2m_ctx_create.argtypes = [ci, P(vp)]
        L.b2m_ctx_destroy.argtypes = [vp]
        L.b2m_ctx_destroy.restype = None
        L.b2m_ctx_launches.argtypes = [vp]
        L.b2m_ctx_launches.restype = ctypes.c_ulonglong
        L.b2m_comm_unique_id.argtypes = [vp, sz]
        L.b2m_ctx_attach_comm.argtypes = [vp, vp, sz, ci, ci]
        L.b2m_ctx_profile.argtypes = [vp, ci]
        L.b2m_ctx_profile_report.argtypes = [vp, ctypes.c_char_p, sz]
        L.b2m_ntt.argtypes = [vp, ci, vp, ctypes.c_uint, ci, ci]
        L.b2m_msm_g1.argtypes = [vp, ci, vp, vp, sz, vp, P(ci)]
        L.b2m_srs_create.argtypes = [vp, ci, vp, sz, vp, vp, sz, ci, P(vp)]
        L.b2m_srs_destroy.argtypes = [vp]
        L.b2m_srs_destroy.restype = None
        L.b2m_srs_size.argtypes = [vp]
        L.b2m_srs_size.restype = sz
        L.b2m_srs_window_bits.argtypes = [vp]
        L.b2m_srs_affine_levels.argtypes = [vp]
        L.b2m_srs_msm.argtypes = [vp, sz, vp, sz, vp, P(ci)]
        L.b2m_g1_powers.argtypes = [vp, ci, vp, vp, sz, vp]
        L.b2m_fixed_base_msm.argtypes = [vp, ci, vp, vp, sz, vp]
        L.b2m_g2_scalar_muls.argtypes = [ci, vp, vp, sz, vp]
        L.b2m_srs_export_g1.argtypes = [vp, sz, sz, vp]
        L.b2m_g1_from_uncompressed.argtypes = [vp, ci, vp, sz, vp]
        L.b2m_g1_to_uncompressed.argtypes = [vp, ci, vp, sz, vp]
        L.b2m_pc_commit.argtypes = [vp, ci, sz, vp, vp, vp, vp, P(Rng), vp, vp, vp, vp, sz]
        L.b2m_pc_open.argtypes = [vp, ci, sz, vp, vp, vp, vp, vp, sz, ctypes.c_int64, vp, vp, vp, P(ci), vp]
        L.b2m_trim.argtypes = [vp, ci, sz, sz, vp, sz, P(vp)]
        L.b2m_ck_destroy.argtypes = [vp]
        L.b2m_ck_destroy.restype = None
        L.b2m_ck_supported_degree.argtypes = [vp]
        L.b2m_ck_supported_degree.restype = sz
        L.b2m_ck_shift_power.argtypes = [vp, u64, vp]
        L.b2m_ck_commit.argtypes = [vp, sz, vp, vp, vp, vp, P(Rng), vp, vp, vp, vp, sz]
        L.b2m_ck_open_combinations.argtypes = [vp, sz, vp, vp, vp, vp, vp, vp, sz, sz, vp, vp, vp, sz, vp, vp, sz, vp, vp, vp, vp, vp]
        if hasattr(L, "b2m_index_create"):
            L.b2m_index_create.argtypes = [vp, ci, sz, sz, sz, P(Matrix), P(Matrix), P(Matrix), P(vp)]
            L.b2m_index_destroy.argtypes = [vp]
            L.b2m_index_destroy.restype = None
            L.b2m_index_vk_bytes.argtypes = [vp, vp, sz, P(sz)]
            L.b2m_index_comms.argtypes = [vp, vp]
            L.b2m_index_stage.argtypes = [vp, vp, sz, vp, sz]
            L.b2m_prove.argtypes = [vp, vp, sz, vp, sz, P(Rng), vp, sz, P(sz)]
            L.b2m_prove_timings.argtypes = [vp, ctypes.c_char_p, sz]
        L.b2m_verifier_create.argtypes = [vp, ci, ci, vp, sz, vp, vp, vp, vp, sz, sz, vp, vp, P(vp)]
        L.b2m_verifier_destroy.argtypes = [vp]
        L.b2m_verifier_destroy.restype = None
        L.b2m_verify.argtypes = [vp, sz, vp, vp, vp, vp, P(Rng), vp]
        L.b2m_verify_timings.argtypes = [vp, ctypes.c_char_p, sz]
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise B2MError(rc, lib().b2m_last_error().decode())


def ptr(a):
    """void* of a C-contiguous numpy array (or None)."""
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(ctypes.c_void_p)


# ---- integer <-> limb-array helpers (host-side marshalling only) ---------------------------
def ints_to_limbs(vals, nlimbs):
    """list of python ints -> (len, nlimbs) uint64 little-endian limbs."""
    out = np.zeros((len(vals), nlimbs), dtype=np.uint64)
    mask = (1 << 64) - 1
    for i, v in enumerate(vals):
        for j in range(nlimbs):
            out[i, j] = (v >> (64 * j)) & mask
    return out


def limbs_to_ints(arr):
    arr = np.asarray(arr, dtype=np.uint64)
    if arr.ndim == 1:
        arr = arr[None, :]
    return [sum(int(row[j]) << (64 * j) for j in range(arr.shape[1])) for row in arr]
