"""ctypes binding of libcandlezip_b200.so (the C ABI declared in include/candlezip_b200.h).

There is no CPU fallback: importing works anywhere the shared library loads, but every compute entry
point returns CZ_ERR_NO_DEVICE without an sm_100 GPU and the wrappers raise `CzError`.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcandlezip_b200.so")

u8p = C.POINTER(C.c_uint8)
u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)
f32p = C.POINTER(C.c_float)
f64p = C.POINTER(C.c_double)
szp = C.POINTER(C.c_size_t)

CZ_OK = 0
CZ_ERR_INVALID = -1
CZ_ERR_NO_DEVICE = -2
CZ_ERR_ZERO_WIDTH = -4
CZ_ERR_UNSUPPORTED = -7
CZ_ERR_SYMBOL_RANGE = -8
CZ_CDF_SMOLLM, CZ_CDF_RWKV_LITERALS, CZ_CDF_SMOLLM_FLOOR = 0, 1, 2
CZ_ARCH_SMOLLM, CZ_ARCH_RWKV7 = 0, 1
CZ_DTYPE_F32, CZ_DTYPE_BF16, CZ_DTYPE_F16 = 0, 1, 2
CZ_ENGINE_TCGEN05, CZ_ENGINE_SIMT = 0, 1
CZ_FLAG_SEGMENTS = 1 << 8
CZ_FLAG_STORED = 1 << 9
CZ_FLAG_PDF_FLOOR = 1 << 10
NO_ZERO_WIDTH = 2 ** 64 - 1  # cz_model_set_zero_width_out: the segment has no zero-width token
K_FAMILIES = ("gemm_qkv", "attn", "elemwise", "cdf", "coder", "other", "gemm_o", "gemm_gu", "gemm_down", "gemm_head", "cdf_prefix")


class CzError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"candlezip_b200 error {code}: {msg}")
        self.code = code


class ModelConfig(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("arch", "vocab", "d_model", "n_layers", "n_heads", "n_kv_heads", "head_dim", "d_ffn")] + [
        ("norm_eps", C.c_float),
        ("rope_theta", C.c_float),
    ] + [(n, C.c_int) for n in ("lora_w", "lora_a", "lora_v", "lora_g", "engine")]


class PrimeEvent(C.Structure):
    _fields_ = [("i", C.c_uint64), ("prime", u32p), ("prime_len", C.c_uint32), ("hold_until", C.c_uint64), ("hist_take", C.c_uint32)]


class Schedule(C.Structure):
    _fields_ = [
        ("context", C.c_uint32),
        ("reprime_interval", C.c_uint32),
        ("n_segments", C.c_uint32),
        ("seg_start", u64p),
        ("bos", C.c_uint32),
        ("events", C.POINTER(PrimeEvent)),
        ("n_events", C.c_uint32),
        ("max_batch_tokens", C.c_uint32),
    ]


class Bitstreams(C.Structure):
    _fields_ = [("data", u8p), ("cap", C.c_size_t), ("seg_off", u64p)]


class XeJob(C.Structure):
    _fields_ = [("prime", u32p), ("prime_len", C.c_uint32), ("targets", u32p), ("n_targets", C.c_uint32)]


class HeaderV2(C.Structure):
    _fields_ = [
        ("bos_token_id", C.c_uint32),
        ("token_count", C.c_uint64),
        ("orig_len_bytes", C.c_uint64),
        ("model_hash16", C.c_uint8 * 16),
        ("tokenizer_hash16", C.c_uint8 * 16),
        ("orig_hash16", C.c_uint8 * 16),
        ("reserved_flags", C.c_uint32),
        ("context_window", C.c_uint32),
        ("vocab_size", C.c_uint32),
        ("model_file_repr_len", C.c_uint32),
        ("reprime_interval", C.c_uint32),
    ]


# every symbol include/candlezip_b200.h declares: (restype, argtypes)
_vp = C.c_void_p
SIGNATURES = {
    "cz_abi_version": (C.c_int, []),
    "cz_init": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "cz_shutdown": (None, [_vp]),
    "cz_last_error": (C.c_char_p, []),
    "cz_launch_count": (C.c_uint64, [_vp]),
    "cz_profile_enable": (C.c_int, [_vp, C.c_int]),
    "cz_ctx_stream": (_vp, [_vp]),
    "cz_profile_read": (C.c_int, [_vp, f64p, u64p, C.c_int]),
    "cz_cdf_bounds": (C.c_int, [_vp, f32p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, u32p, u32p, u32p]),
    "cz_cdf_bounds_dev": (C.c_int, [_vp, _vp, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, _vp, _vp, _vp]),
    "cz_cdf_search": (C.c_int, [_vp, f32p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, u32p, u32p, u32p, u32p]),
    "cz_cdf_full": (C.c_int, [_vp, f32p, C.c_size_t, C.c_int, u32p]),
    "cz_xe_bits_cols": (C.c_int, [_vp, f32p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, u32p, f64p]),
    "cz_ac_encode_lanes": (C.c_int, [_vp, u32p, u32p, u64p, C.c_size_t, u8p, u64p, u64p]),
    "cz_ac_decode_lanes": (C.c_int, [_vp, u8p, u64p, u64p, u64p, C.c_size_t, u32p, C.c_size_t, u32p]),
    "cz_model_config_smollm_135m": (None, [C.POINTER(ModelConfig)]),
    "cz_model_config_rwkv7_0p1b": (None, [C.POINTER(ModelConfig)]),
    "cz_model_create": (C.c_int, [_vp, C.POINTER(ModelConfig), C.POINTER(_vp)]),
    "cz_model_free": (None, [_vp]),
    "cz_model_set_tensor": (C.c_int, [_vp, C.c_char_p, _vp, C.c_int, C.c_size_t]),
    "cz_model_get_tensor": (C.c_int, [_vp, C.c_char_p, f32p, C.c_size_t]),
    "cz_model_tensor_count": (C.c_int, [_vp]),
    "cz_model_tensor_info": (C.c_int, [_vp, C.c_int, C.POINTER(C.c_char_p), szp]),
    "cz_model_random_init": (C.c_int, [_vp, C.c_uint64, C.c_float, C.c_float]),
    "cz_model_load_safetensors": (C.c_int, [_vp, C.POINTER(C.c_char_p), C.c_int]),
    "cz_model_config_get": (C.c_int, [_vp, C.POINTER(ModelConfig)]),
    "cz_session_new": (C.c_int, [_vp, C.POINTER(_vp)]),
    "cz_session_free": (None, [_vp]),
    "cz_session_vocab_size": (C.c_size_t, [_vp]),
    "cz_session_max_context_length": (C.c_size_t, [_vp]),
    "cz_session_index_pos": (C.c_size_t, [_vp]),
    "cz_session_step_logits": (C.c_int, [_vp, C.c_uint32, f32p]),
    "cz_session_reprime": (C.c_int, [_vp, u32p, C.c_size_t, f32p]),
    "cz_encode": (C.c_int, [_vp, u32p, C.c_size_t, C.POINTER(Schedule), C.POINTER(Bitstreams)]),
    "cz_decode": (C.c_int, [_vp, u8p, u64p, C.c_size_t, C.POINTER(Schedule), u32p]),
    "cz_encode_dev": (C.c_int, [_vp, _vp, C.c_size_t, C.POINTER(Schedule), _vp, C.c_size_t, u64p]),
    "cz_model_set_digest_out": (C.c_int, [_vp, u8p, C.c_size_t]),
    "cz_model_set_pdf_floor": (C.c_int, [_vp, C.c_int]),
    "cz_model_set_zero_width_out": (C.c_int, [_vp, u64p, C.c_size_t]),
    "cz_xe_bits": (C.c_int, [_vp, C.POINTER(XeJob), C.c_size_t, f64p]),
    "cz_chunk_logits": (C.c_int, [_vp, u32p, C.c_size_t, u32p, C.c_size_t, f32p]),
    "cz_container_header_size": (C.c_size_t, [C.POINTER(HeaderV2)]),
    "cz_container_write_header": (C.c_size_t, [u8p, C.c_size_t, C.POINTER(HeaderV2), u8p]),
    "cz_container_read_header": (C.c_size_t, [u8p, C.c_size_t, C.POINTER(HeaderV2), szp]),
    "cz_container_write_gates": (C.c_size_t, [u8p, C.c_size_t, u8p, C.c_size_t]),
    "cz_container_read_gates": (C.c_size_t, [u8p, C.c_size_t, u8p, C.c_size_t, szp]),
    "cz_container_write_segments": (C.c_size_t, [u8p, C.c_size_t, C.c_int, u64p, u64p, C.c_size_t]),
    "cz_container_read_segments": (C.c_size_t, [u8p, C.c_size_t, C.POINTER(C.c_int), u64p, u64p, C.c_size_t, szp]),
    "cz_flags_pack": (C.c_uint32, [C.c_int, C.c_int, C.c_int, C.c_uint32]),
    "cz_blake3_16": (None, [u8p, C.c_size_t, u8p]),
    "cz_test_gemm": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_uint16), C.POINTER(C.c_uint16), C.c_int, C.c_int, _vp,
                              C.c_int]),
    "cz_test_gemm_norm": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_uint16), C.POINTER(C.c_uint16), C.POINTER(C.c_uint16),
                                   C.POINTER(C.c_float), C.c_float, C.POINTER(C.c_float), C.POINTER(C.c_uint16), C.POINTER(C.c_float),
                                   C.POINTER(C.c_uint16)]),
    "cz_test_attention": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_uint16), C.POINTER(C.c_uint16), C.POINTER(C.c_uint16), C.c_int,
                                   C.POINTER(C.c_uint16)]),
    "cz_test_expf_exhaustive": (C.c_int, [_vp, u64p, u64p, u64p]),
    "cz_test_div_random": (C.c_int, [_vp, C.c_uint64, C.c_uint64, u64p]),
    "cz_test_cdf_ecache_state": (C.c_int, [_vp, C.POINTER(C.c_int), u64p]),
    "cz_schedule_chunks": (C.c_size_t, [C.c_uint64, C.c_uint32, C.c_uint32, u64p, u32p, u64p, u32p, C.c_size_t]),
}


def load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(make -C candlezip_b200/csrc). There is no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here == the library does not export what the header declares
        fn.restype = res
        fn.argtypes = args
    return lib


lib = load()


def check(rc):
    if rc != CZ_OK:
        raise CzError(rc, lib.cz_last_error().decode(errors="replace"))
