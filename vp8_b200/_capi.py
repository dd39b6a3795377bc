"""ctypes binding of libvp8r.so (include/vp8r.h).  Plain C types only; no torch objects cross it."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VP8R_LIB") or os.path.join(_HERE, "_lib", "libvp8r.so")  # VP8R_LIB: development builds


class MbInfo(C.Structure):
    _fields_ = [("flags", C.c_uint32), ("coef_mask", C.c_uint32), ("coef_offset", C.c_uint32),
                ("mv", C.c_int16 * 2), ("aux", C.c_uint32 * 2), ("reserved", C.c_uint32 * 2)]


class FrameHdr(C.Structure):
    _fields_ = [("width", C.c_uint16), ("height", C.c_uint16), ("mb_cols", C.c_uint16), ("mb_rows", C.c_uint16),
                ("key_frame", C.c_uint8), ("version", C.c_uint8), ("show_frame", C.c_uint8),
                ("filter_type", C.c_uint8), ("loop_filter_level", C.c_uint8), ("sharpness_level", C.c_uint8),
                ("refresh_last", C.c_uint8), ("refresh_golden", C.c_uint8), ("refresh_altref", C.c_uint8),
                ("copy_to_golden", C.c_uint8), ("copy_to_altref", C.c_uint8),
                ("sign_bias_golden", C.c_uint8), ("sign_bias_altref", C.c_uint8), ("q_index", C.c_uint8),
                ("modes_deferred", C.c_uint8), ("tokens_deferred", C.c_uint8),
                ("dq", (C.c_int16 * 6) * 4),
                ("n_coef_blocks", C.c_uint32), ("n_payload_blocks", C.c_uint32),
                ("n_inter_mbs", C.c_uint32), ("n_split_mbs", C.c_uint32),
                ("n_intra_levels", C.c_uint32), ("intra_levels_at", C.c_uint32), ("tokens_at", C.c_uint32), ("modes_at", C.c_uint32)]


class TokenHdr(C.Structure):
    _fields_ = [("n_parts", C.c_uint32), ("part_off", C.c_uint32 * 8), ("part_size", C.c_uint32 * 8),
                ("raw_bytes", C.c_uint32), ("reserved", C.c_uint32 * 6), ("coef_probs", C.c_uint8 * 1056)]


class FrameDesc(C.Structure):
    _fields_ = [("hdr", FrameHdr), ("mbs", C.POINTER(MbInfo)), ("payload", C.POINTER(C.c_int16))]


class Timers(C.Structure):
    _fields_ = [("ms_inter", C.c_double), ("ms_intra", C.c_double), ("ms_filter", C.c_double),
                ("ms_h2d", C.c_double), ("ms_d2h", C.c_double), ("ms_tokens", C.c_double),
                ("launches_inter", C.c_uint64), ("launches_intra", C.c_uint64), ("launches_filter", C.c_uint64),
                ("launches_other", C.c_uint64), ("frames", C.c_uint64), ("coef_blocks", C.c_uint64),
                ("alg_bytes", C.c_uint64), ("ms_border", C.c_double)]


# name -> (restype, argtypes); mirrors include/vp8r.h one to one (tests check the two agree).
SIGNATURES = {
    "vp8r_parser_create": (C.c_void_p, []),
    "vp8r_parser_destroy": (None, [C.c_void_p]),
    "vp8r_parser_reset": (None, [C.c_void_p]),
    "vp8r_parser_set_defer_tokens": (None, [C.c_void_p, C.c_int]),
    "vp8r_parser_set_defer_modes": (None, [C.c_void_p, C.c_int]),
    "vp8r_frame_create": (C.c_void_p, [C.c_int]),
    "vp8r_frame_destroy": (None, [C.c_void_p]),
    "vp8r_frame_get_desc": (C.c_int, [C.c_void_p, C.POINTER(FrameDesc)]),
    "vp8r_parser_parse": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "vp8r_parse_batch": (C.c_int, [C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_size_t),
                                   C.POINTER(C.c_void_p), C.c_int, C.POINTER(C.c_int)]),
    "vp8r_is_key_frame": (C.c_int, [C.c_void_p, C.c_size_t]),
    "vp8r_engine_create": (C.c_int, [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]),
    "vp8r_engine_destroy": (None, [C.c_void_p]),
    "vp8r_engine_sync": (C.c_int, [C.c_void_p]),
    "vp8r_engine_fence": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64)]),
    "vp8r_engine_wait": (C.c_int, [C.c_void_p, C.c_uint64]),
    "vp8r_stream_open": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "vp8r_stream_close": (None, [C.c_void_p]),
    "vp8r_frame_upload": (C.c_int, [C.c_void_p, C.c_void_p]),
    "vp8r_frame_release_host": (C.c_int, [C.c_void_p]),
    "vp8r_reconstruct_batch": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    "vp8r_stream_frame_bytes": (C.c_size_t, [C.c_void_p]),
    "vp8r_stream_dims": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "vp8r_read_batch": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                  C.POINTER(C.c_size_t), C.c_int]),
    "vp8r_read_batch_packed": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.c_void_p, C.c_size_t, C.c_int]),
    "vp8r_encode_key_frames": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int,
                                         C.c_int, C.c_int, C.c_uint, C.POINTER(C.c_void_p)]),
    "vp8r_encode_inter_frames": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int, C.c_int,
                                           C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "vp8r_encode_key_frames_device": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.c_void_p, C.c_size_t, C.c_int,
                                                C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint,
                                                C.POINTER(C.c_void_p)]),
    "vp8r_encode_inter_frames_device": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.c_void_p, C.c_size_t, C.c_int,
                                                  C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                                  C.POINTER(C.c_void_p)]),
    "vp8r_convert_to_i420_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_int,
                                              C.c_void_p, C.c_size_t, C.c_void_p]),
    "vp8r_frame_write_bitstream": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]),
    "vp8r_frame_write_bitstream_in": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]),
    "vp8r_read_batch_packed_as": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.c_void_p, C.c_size_t, C.c_int, C.c_int]),
    "vp8r_read_batch_device": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.c_void_p, C.c_size_t, C.c_int,
                                         C.c_void_p]),
    "vp8r_stream_read_frame": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "vp8r_stream_checksum": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64)]),
    "vp8r_checksum_batch": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]),
    "vp8r_checksum_i420": (C.c_uint64, [C.c_void_p, C.c_int, C.c_int]),
    "vp8r_stream_decode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_int)]),
    "vp8r_engine_set_timing": (C.c_int, [C.c_void_p, C.c_int]),
    "vp8r_engine_get_timers": (C.c_int, [C.c_void_p, C.POINTER(Timers), C.c_int]),
    "vp8r_last_error": (C.c_char_p, []),
    "vp8r_version": (C.c_char_p, []),
    "vp8r_has_cuda": (C.c_int, []),
}

_lib = None


def load():
    """Loads libvp8r.so.  Fails loudly when it has not been built: there is no Python/CPU fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run ./build.sh (or __graft_entry__.build()) first; "
                           "vp8_b200 has no fallback implementation")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class Vp8rError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"vp8r error {code}: {msg}")
        self.code = code


def check(rc):
    if rc != 0:
        raise Vp8rError(rc, (load().vp8r_last_error() or b"").decode())
