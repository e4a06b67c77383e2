"""ctypes binding of libcapycrypt_gpu.so (C ABI declared in include/capy_gpu.h).

There is no CPU fallback: if the shared library is missing or fails to load, importing this
module raises (build it with `python -m capycrypt_b200.build`).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CAPY_GPU_LIB", os.path.join(_HERE, "_lib", "libcapycrypt_gpu.so"))

OK = 0
ERR_BAD_SECPARAM = -1
ERR_BAD_ARG = -2
ERR_CUDA = -3
ERR_BAD_POINT = -4
ERR_NO_DEVICE = -5
ERR_OOM = -6
AE_SHA3 = 0
AE_KEM = 1

u8p = C.c_void_p  # raw addresses (host numpy buffers or device pointers)
u64p = C.c_void_p
vp = C.c_void_p
i32 = C.c_int
u32 = C.c_uint32
u64 = C.c_uint64

# every symbol include/capy_gpu.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "capy_gpu_init": (i32, [C.POINTER(C.c_int), i32, C.POINTER(vp)]),
    "capy_gpu_destroy": (None, [vp]),
    "capy_gpu_device_count": (i32, [vp]),
    "capy_gpu_scrub": (i32, [vp]),
    "capy_strerror": (C.c_char_p, [i32]),
    "capy_last_cuda_error": (C.c_char_p, [vp]),
    "capy_version": (i32, []),
    "capy_host_alloc": (vp, [C.c_size_t]),
    "capy_host_free": (None, [vp]),
    "capy_launch_count": (u64, [vp]),
    "capy_copy_probe": (i32, [vp, i32, vp, C.c_size_t, vp, C.c_size_t, i32, C.POINTER(C.c_double)]),
    "capy_plan_tiers": (i32, [vp, u32, u64, u32, u64, i32, vp, vp]),
    "capy_plan_tiers3": (i32, [vp, u32, u64, u32, u64, i32, vp, vp]),
    "capy_gpu_set_plan_cache": (i32, [vp, i32]),
    "capy_lpt_shares": (i32, [vp, u64, u32, u32, u64, vp]),
    "capy_chain_cut": (i32, [i32, u64, u64, u64, vp]),
    "capy_sha3_batch": (i32, [vp, i32, u8p, u64p, u64, u8p, u32]),
    "capy_sha3_batch_fixed": (i32, [vp, i32, u8p, u64, u64, u64, u8p, u32]),
    "capy_sha3_batch_dev": (i32, [vp, i32, vp, i32, u8p, u64p, u64, u8p, u32]),
    "capy_sha3_batch_fixed_dev": (i32, [vp, i32, vp, i32, u8p, u64, u64, u64, u8p, u32]),
    "capy_cshake_batch": (i32, [vp, i32, u8p, u64p, u64, u8p, u32, u8p, u32, u64, u8p]),
    "capy_cshake_batch_dev": (i32, [vp, i32, vp, i32, u8p, u64p, u64, u8p, u32, u8p, u32, u64, u8p]),
    "capy_kmac_xof_batch": (i32, [vp, i32, u8p, u64p, u8p, u64p, u64, u8p, u32, u64, u64p, u8p]),
    "capy_kmac_xof_batch_dev": (i32, [vp, i32, vp, i32, u8p, u64p, u8p, u64p, u64, u8p, u32, u64, u64p, u8p]),
    "capy_kmac_xof_batch_fixed_dev": (i32, [vp, i32, vp, i32, u8p, u64, u64, u8p, u64, u64, u64, u8p, u32, u64, u8p]),
    "capy_fips_shake_batch_dev": (i32, [vp, i32, vp, i32, u8p, u64p, u64, u64, u8p]),
    "capy_ed448_fixed_base_batch": (i32, [vp, u8p, u64, u8p]),
    "capy_ed448_fixed_base_batch_dev": (i32, [vp, i32, vp, u8p, u64, u8p]),
    "capy_ed448_var_base_batch": (i32, [vp, u8p, u8p, u64, u8p]),
    "capy_ed448_var_base_batch_dev": (i32, [vp, i32, vp, u8p, u8p, u64, u8p, vp]),
    "capy_ed448_keygen_batch": (i32, [vp, i32, u8p, u64p, u64, u8p]),
    "capy_ed448_keygen_batch_dev": (i32, [vp, i32, vp, i32, u8p, u64p, u64, u8p]),
    "capy_ed448_sign_batch": (i32, [vp, i32, u8p, u64p, u8p, u64p, u64, u8p, u8p]),
    "capy_ed448_sign_batch_dev": (i32, [vp, i32, vp, i32, u8p, u64p, u8p, u64p, u64, u8p, u8p]),
    "capy_ed448_verify_batch": (i32, [vp, i32, u8p, u8p, u64p, u8p, u8p, u64, u8p]),
    "capy_ed448_verify_batch_dev": (i32, [vp, i32, vp, i32, u8p, u8p, u64p, u8p, u8p, u64, u8p, vp]),
    "capy_ed448_ecdh_batch": (i32, [vp, u8p, u8p, u64, u8p, u8p]),
    "capy_sponge_encrypt_batch": (i32, [vp, i32, i32, u8p, u64p, u8p, u64, u8p, u64p, u64, u8p, u8p]),
    "capy_sponge_decrypt_batch": (i32, [vp, i32, i32, u8p, u64p, u8p, u64, u8p, u64p, u8p, u64, u8p, u8p]),
    "capy_sponge_encrypt_batch_dev": (i32, [vp, i32, vp, i32, i32, u8p, u64p, u64, u8p, u64, u8p, u64p, u64, u8p, u8p]),
    "capy_sponge_decrypt_batch_dev": (i32, [vp, i32, vp, i32, i32, u8p, u64p, u64, u8p, u64, u8p, u64p, u8p, u64, u8p,
                                            u8p]),
    "capy_ed448_key_encrypt_batch": (i32, [vp, i32, u8p, u8p, u8p, u64p, u64, u8p, u8p, u8p]),
    "capy_ed448_key_decrypt_batch": (i32, [vp, i32, u8p, u64p, u8p, u8p, u64p, u8p, u64, u8p, u8p]),
    "capy_ed448_key_encrypt_batch_dev": (i32, [vp, i32, vp, i32, u8p, u8p, u8p, u64p, u64, u8p, u8p, u8p, vp]),
    "capy_ed448_key_decrypt_batch_dev": (i32, [vp, i32, vp, i32, u8p, u64p, u8p, u8p, u64p, u8p, u64, u8p, u8p, vp]),
    "capy_ed448_pub_prepare": (i32, [vp, u8p, C.POINTER(vp)]),
    "capy_ed448_pub_uses_comb": (i32, [vp]),
    "capy_ed448_pub_free": (None, [vp]),
    "capy_ed448_verify_prepared_batch": (i32, [vp, i32, vp, u8p, u64p, u8p, u8p, u64, u8p]),
    "capy_ed448_verify_prepared_batch_dev": (i32, [vp, i32, vp, i32, vp, u8p, u64p, u8p, u8p, u64, u8p]),
    "capy_ed448_key_encrypt_prepared_batch": (i32, [vp, i32, vp, u8p, u8p, u64p, u64, u8p, u8p, u8p]),
    "capy_ed448_key_encrypt_prepared_batch_dev": (i32, [vp, i32, vp, i32, vp, u8p, u8p, u64p, u64, u8p, u8p, u8p]),
    "capy_sha3_hasher_new": (i32, [vp, i32, u64, C.POINTER(vp)]),
    "capy_kmac_xof_hasher_new": (i32, [vp, i32, u8p, u64p, u64, u8p, u32, C.POINTER(vp)]),
    "capy_hasher_device_range": (i32, [vp, i32, C.POINTER(u64), C.POINTER(u64)]),
    "capy_hasher_update": (i32, [vp, vp, u8p, u64p]),
    "capy_hasher_update_dev": (i32, [vp, vp, i32, vp, u8p, u64p]),
    "capy_hasher_final": (i32, [vp, vp, u64, u64p, u8p]),
    "capy_hasher_final_dev": (i32, [vp, vp, i32, vp, u64, u64p, u8p]),
    "capy_hasher_free": (None, [vp]),
    "capy_sponge_encrypt_stream_new": (i32, [vp, i32, i32, u8p, u64p, u8p, u64, u64, C.POINTER(vp)]),
    "capy_ed448_key_encrypt_stream_new": (i32, [vp, i32, u8p, vp, u8p, u64, u8p, C.POINTER(vp)]),
    "capy_ed448_verify_stream_new": (i32, [vp, i32, u8p, vp, u8p, u8p, u64, C.POINTER(vp)]),
    "capy_hasher_encrypt_update": (i32, [vp, vp, u8p, u64p, u8p]),
    "capy_hasher_encrypt_update_dev": (i32, [vp, vp, i32, vp, u8p, u64p, u8p]),
    "capy_hasher_verify_final": (i32, [vp, vp, u8p]),
    "capy_hasher_verify_final_dev": (i32, [vp, vp, i32, vp, u8p, vp]),
    "capy_ed448_sign_stream_new": (i32, [vp, i32, u8p, u64p, u64, C.POINTER(vp)]),
    "capy_sponge_decrypt_stream_new": (i32, [vp, i32, i32, u8p, u64p, u8p, u64, u8p, u64, C.POINTER(vp)]),
    "capy_ed448_key_decrypt_stream_new": (i32, [vp, i32, u8p, u64p, u8p, u8p, u64, C.POINTER(vp)]),
    "capy_hasher_next_pass": (i32, [vp, vp, u8p]),
    "capy_hasher_next_pass_dev": (i32, [vp, vp, i32, vp, u8p, vp]),
    "capy_hasher_decrypt_update": (i32, [vp, vp, u8p, u64p, u8p]),
    "capy_hasher_decrypt_update_dev": (i32, [vp, vp, i32, vp, u8p, u64p, u8p]),
    "capy_hasher_decrypt_final": (i32, [vp, vp, u8p]),
    "capy_hasher_decrypt_final_dev": (i32, [vp, vp, i32, vp, u8p, vp]),
    "capy_hasher_sign_final": (i32, [vp, vp, u8p, u8p, u8p]),
    "capy_hasher_sign_final_dev": (i32, [vp, vp, i32, vp, u8p, u8p, u8p]),
    "capy_hasher_export_size": (i32, [vp, C.POINTER(u64)]),
    "capy_hasher_export": (i32, [vp, vp, u8p, u64]),
    "capy_hasher_blob_info": (i32, [u8p, u64, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(u64)]),
    "capy_hasher_import": (i32, [vp, u8p, u64, C.POINTER(vp)]),
    "capy_hasher_fork": (i32, [vp, vp, u64p, u64, C.POINTER(vp)]),
}


def declared_symbols(header_path: str | None = None) -> list[str]:
    """Function names declared in include/capy_gpu.h (parsed, so tests can diff vs SIGNATURES)."""
    import re

    header_path = header_path or os.path.join(_HERE, "..", "include", "capy_gpu.h")
    src = open(header_path).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(capy_[a-z0-9_]+)\s*\(", src)))


def load(path: str | None = None) -> C.CDLL:
    path = path or LIB_PATH
    if not os.path.exists(path):
        raise ImportError(
            f"libcapycrypt_gpu.so not found at {path}: the CUDA engine is required (no CPU fallback). "
            "Build it with `python -m capycrypt_b200.build`."
        )
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    return lib


class CapyError(RuntimeError):
    def __init__(self, status: int, msg: str):
        super().__init__(f"capy_gpu status {status}: {msg}")
        self.status = status
