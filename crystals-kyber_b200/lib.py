"""ctypes binding of libmlkem_b200.so (include/mlkem_b200.h).  Fails loudly when the library is absent."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libmlkem_b200.so")

MEM_HOST, MEM_DEVICE = 0, 1
FLAG_FIPS203 = 1


class MlKemB200Error(RuntimeError):
    pass


class Opts(C.Structure):
    _fields_ = [("device", C.c_int), ("mem", C.c_int), ("stream", C.c_void_p), ("chunk_items", C.c_int),
                ("sample_group_limit", C.c_int), ("flags", C.c_int)]


_lib = None

# every symbol include/mlkem_b200.h declares: name -> (restype, argtypes)
_P8, _P16, _PO = C.c_void_p, C.c_void_p, C.POINTER(Opts)
SIGNATURES = {
    "mlkem_b200_version": (C.c_char_p, []),
    "mlkem_b200_last_error": (C.c_char_p, []),
    "mlkem_b200_launch_count": (C.c_ulonglong, []),
    "mlkem_b200_device_count": (C.c_int, []),
    "mlkem_b200_synchronize": (C.c_int, [C.c_int, C.c_void_p]),
    "mlkem_b200_host_alloc": (C.c_void_p, [C.c_size_t]),
    "mlkem_b200_host_alloc_wc": (C.c_void_p, [C.c_size_t]),
    "mlkem_b200_host_free": (None, [C.c_void_p]),
    "mlkem_b200_copy_probe": (C.c_int, [C.c_size_t, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_int, C.POINTER(C.c_void_p),
                                        C.POINTER(C.c_size_t), _PO]),
    "mlkem_b200_release": (None, [C.c_int]),
    "mlkem_b200_ek_bytes": (C.c_uint, [C.c_int]),
    "mlkem_b200_dk_bytes": (C.c_uint, [C.c_int]),
    "mlkem_b200_dkpke_bytes": (C.c_uint, [C.c_int]),
    "mlkem_b200_ct_bytes": (C.c_uint, [C.c_int]),
    "mlkem_b200_keygen_batch": (C.c_int, [C.c_int, C.c_size_t, _P8, _P8, _P8, _P8, _PO]),
    "mlkem_b200_encaps_batch": (C.c_int, [C.c_int, C.c_size_t, _P8, _P8, _P8, _P8, _PO]),
    "mlkem_b200_decaps_batch": (C.c_int, [C.c_int, C.c_size_t, _P8, _P8, _P8, _PO]),
    "mlkem_b200_check_dk_batch": (C.c_int, [C.c_int, C.c_size_t, _P8, C.c_void_p, _PO]),
    "mlkem_b200_keygen_cells_batch": (C.c_int, [C.c_int, C.c_size_t, _P8, _P8, _P8, _P8, _PO]),
    "mlkem_b200_encaps_cells_batch": (C.c_int, [C.c_int, C.c_size_t, _P8, _P8, _P8, _P8, _PO]),
    "mlkem_b200_decaps_cells_batch": (C.c_int, [C.c_int, C.c_size_t, _P8, _P8, _P8, _PO]),
    "mlkem_b200_cells_from_bytes": (C.c_int, [C.c_size_t, _P8, C.c_void_p, _PO]),
    "mlkem_b200_cells_to_bytes": (C.c_int, [C.c_size_t, C.c_void_p, _P8, _PO]),
    "mlkem_b200_keys_load": (C.c_int, [C.c_int, C.c_size_t, _P8, C.c_void_p, _PO, C.POINTER(C.c_void_p)]),
    "mlkem_b200_keys_load_ek": (C.c_int, [C.c_int, C.c_size_t, _P8, _PO, C.POINTER(C.c_void_p)]),
    "mlkem_b200_keys_from_seeds": (C.c_int, [C.c_int, C.c_size_t, _P8, _P8, _PO, C.POINTER(C.c_void_p)]),
    "mlkem_b200_keys_count": (C.c_size_t, [C.c_void_p]),
    "mlkem_b200_keys_free": (None, [C.c_void_p]),
    "mlkem_b200_keys_replace": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, _P8, C.c_void_p, _PO]),
    "mlkem_b200_keys_replace_ek": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, _P8, _PO]),
    "mlkem_b200_keys_replace_from_seeds": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, _P8, _P8, _PO]),
    "mlkem_b200_keys_export_ek": (C.c_int, [C.c_void_p, C.c_size_t, C.c_size_t, _P8, _PO]),
    "mlkem_b200_encaps_keyed_batch": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, _P8, _P8, _P8, _PO]),
    "mlkem_b200_decaps_keyed_batch": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, _P8, _P8, _PO]),
    "mlkem_b200_kem_keygen_batch": (C.c_int, [C.c_int, C.c_size_t, _P8, _P8, _PO]),
    "mlkem_b200_kem_encaps_batch": (C.c_int, [C.c_int, C.c_size_t, _P8, C.c_size_t, _P8, _P8, _PO]),
    "mlkem_b200_kem_decaps_batch": (C.c_int, [C.c_int, C.c_size_t, _P8, C.c_size_t, _P8, C.c_size_t, _P8, C.c_void_p, _PO]),
    "mlkem_b200_kem_keygen_seeded_batch": (C.c_int, [C.c_int, C.c_size_t, _P8, _P8, _P8, _PO]),
    "mlkem_b200_kem_encaps_seeded_batch": (C.c_int, [C.c_int, C.c_size_t, _P8, C.c_size_t, _P8, _P8, _P8, _PO]),
    "mlkem_b200_kem_encaps_keyed_batch": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, _P8, _P8, _P8, _PO]),
    "mlkem_b200_keys_generate": (C.c_int, [C.c_int, C.c_size_t, _P8, _PO, C.POINTER(C.c_void_p)]),
    "mlkem_b200_keys_replace_generate": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, _P8, _PO]),
    "mlkem_b200_pke_keygen_batch": (C.c_int, [C.c_int, C.c_size_t, _P8, _P8, _P8, _PO]),
    "mlkem_b200_pke_encrypt_batch": (C.c_int, [C.c_int, C.c_size_t, _P8, _P8, _P8, _P8, _PO]),
    "mlkem_b200_pke_decrypt_batch": (C.c_int, [C.c_int, C.c_size_t, _P8, C.c_size_t, _P8, _P8, _PO]),
    "mlkem_b200_ntt_batch": (C.c_int, [C.c_size_t, _P16, _P16, _PO]),
    "mlkem_b200_intt_batch": (C.c_int, [C.c_size_t, _P16, _P16, _PO]),
    "mlkem_b200_multiply_ntts_batch": (C.c_int, [C.c_size_t, _P16, _P16, _P16, _PO]),
    "mlkem_b200_poly_add_batch": (C.c_int, [C.c_size_t, _P16, _P16, _P16, _PO]),
    "mlkem_b200_poly_sub_batch": (C.c_int, [C.c_size_t, _P16, _P16, _P16, _PO]),
    "mlkem_b200_vector_multiply_batch": (C.c_int, [C.c_int, C.c_size_t, _P16, _P16, _P16, _PO]),
    "mlkem_b200_sample_ntt_batch": (C.c_int, [C.c_size_t, _P8, _P16, _P8, _PO]),
    "mlkem_b200_cbd_batch": (C.c_int, [C.c_int, C.c_size_t, _P8, _P16, _PO]),
    "mlkem_b200_prf_cbd_batch": (C.c_int, [C.c_int, C.c_size_t, _P8, _P8, _P16, _PO]),
    "mlkem_b200_byte_encode_batch": (C.c_int, [C.c_int, C.c_size_t, _P16, _P8, _PO]),
    "mlkem_b200_byte_decode_batch": (C.c_int, [C.c_int, C.c_size_t, _P8, _P16, _PO]),
    "mlkem_b200_compress_batch": (C.c_int, [C.c_int, C.c_size_t, _P16, _P16, _PO]),
    "mlkem_b200_decompress_batch": (C.c_int, [C.c_int, C.c_size_t, _P16, _P16, _PO]),
    "mlkem_b200_compress_encode_batch": (C.c_int, [C.c_int, C.c_size_t, _P16, _P8, _PO]),
    "mlkem_b200_decode_decompress_batch": (C.c_int, [C.c_int, C.c_size_t, _P8, _P16, _PO]),
    "mlkem_b200_hash_batch": (C.c_int, [C.c_int, C.c_size_t, C.c_size_t, _P8, _P8, _PO]),
    "mlkem_b200_sha3_bits_batch": (C.c_int, [C.c_size_t, _P8, C.c_size_t, C.c_void_p, C.c_uint, C.c_size_t, _P8, _PO]),
    "mlkem_b200_tables": (C.c_int, [C.c_void_p, C.c_void_p]),
    "mlkem_b200_profile": (None, [C.c_int]),
    "mlkem_b200_set_streams": (None, [C.c_int]),
    "mlkem_b200_profile_report": (C.c_int, [C.c_char_p, C.c_int]),
    "mlkem_b200_int32_peak": (C.c_int, [C.POINTER(C.c_double)]),
}
# the reference-signature API of include/ml_kem.h (checked for presence only from Python)
COMPAT_SYMBOLS = ["ml_errno", "init", "KEM_KeyGen", "KEM_Encaps", "KEM_Decaps", "SampleNTT", "SamplePolyCBD", "NTT",
                  "InverseNTT", "BitRev7", "BitsToBytes", "BytesToBits", "Compress", "Decompress", "ByteEncode",
                  "ByteDecode", "BaseCaseMultiply", "MultiplyNTTs", "PKE_KeyGen", "PKE_Encrypt", "PKE_Decrypt",
                  "KeyGen_internal", "Encaps_internal", "Decaps_internal", "h2b", "b2h", "sha3_b", "sha3_h", "sha3_s"]


def load(path: str = None):
    """Load libmlkem_b200.so.  No fallback: a missing library is an error.  MLKEM_B200_LIB names another build of the
    same library (the A/B and experiment builds of tools/)."""
    global _lib
    if _lib is not None:
        return _lib
    if path is None:
        path = os.path.abspath(os.environ["MLKEM_B200_LIB"]) if os.environ.get("MLKEM_B200_LIB") else LIB_PATH
    if not os.path.exists(path):
        raise MlKemB200Error(
            f"{path} not found: build it with `make lib` (nvcc, sm_100a). There is no CPU fallback.")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the ABI is incomplete
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
