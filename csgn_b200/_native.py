"""ctypes binding of libcsgn.so (include/csgn.h).  Fails loudly when the CUDA
library is missing or no B200 is visible -- there is no CPU fallback to fall to."""
import ctypes
import os
import re
import warnings

from . import build as _build

_u64 = ctypes.c_uint64
_u64p = ctypes.POINTER(ctypes.c_uint64)
_vp = ctypes.c_void_p
_vpp = ctypes.POINTER(ctypes.c_void_p)

# name -> (restype, argtypes); must cover every function declared in include/csgn.h
SIGNATURES = {
    "csgn_init": (ctypes.c_int, [ctypes.c_int]),
    "csgn_shutdown": (ctypes.c_int, []),
    "csgn_is_initialized": (ctypes.c_int, []),
    "csgn_last_error": (ctypes.c_char_p, []),
    "csgn_version": (ctypes.c_char_p, []),
    "csgn_device_info": (ctypes.c_int, [ctypes.POINTER(ctypes.c_int), _u64p, _u64p, ctypes.POINTER(ctypes.c_int)]),
    "csgn_set_stream": (ctypes.c_int, [_vp]),
    "csgn_get_stream": (_vp, []),
    "csgn_set_auto_lanes": (ctypes.c_int, [ctypes.c_int]),
    "csgn_get_auto_lanes": (ctypes.c_int, []),
    "csgn_sync": (ctypes.c_int, []),
    "csgn_launch_count": (_u64, []),
    "csgn_words_per_block": (ctypes.c_uint32, [_u64]),
    "csgn_host_alloc": (ctypes.c_int, [ctypes.c_size_t, _vpp]),
    "csgn_host_free": (ctypes.c_int, [_vp]),
    "csgn_buf_upload": (ctypes.c_int, [_vp, _u64, ctypes.c_uint32, _vpp]),
    "csgn_buf_upload_copy": (ctypes.c_int, [_vp, _u64, ctypes.c_uint32, _vpp]),
    "csgn_buf_upload_batch": (ctypes.c_int, [_vp, _vp, ctypes.c_uint32, ctypes.c_uint32, _vp]),
    "csgn_buf_free_batch": (ctypes.c_int, [_vp, ctypes.c_uint32]),
    "csgn_buf_alloc": (ctypes.c_int, [_u64, ctypes.c_uint32, _vpp]),
    "csgn_buf_wrap": (ctypes.c_int, [_vp, _u64, ctypes.c_uint32, _vpp]),
    "csgn_buf_clone": (ctypes.c_int, [_vp, _vpp]),
    "csgn_buf_download": (ctypes.c_int, [_vp, _vp]),
    "csgn_buf_download_range": (ctypes.c_int, [_vp, _u64, _u64, _vp]),
    "csgn_buf_slice": (ctypes.c_int, [_vp, _u64, _u64, _vpp]),
    "csgn_buf_free": (ctypes.c_int, [_vp]),
    "csgn_buf_blocks": (_u64, [_vp]),
    "csgn_buf_words_per_block": (ctypes.c_uint32, [_vp]),
    "csgn_buf_device_ptr": (_vp, [_vp]),
    "csgn_mul": (ctypes.c_int, [_vp, _vp, _vpp]),
    "csgn_mul_into": (ctypes.c_int, [_vp, _vp, _vp]),
    "csgn_concat": (ctypes.c_int, [_vp, _vp, _vpp]),
    "csgn_append": (ctypes.c_int, [_vp, _vp]),
    "csgn_concat_lazy": (ctypes.c_int, [_vp, _vp, _vpp]),
    "csgn_buf_segments": (ctypes.c_int, [_vp]),
    "csgn_buf_retained": (ctypes.c_int, [_vp]),
    "csgn_buf_flatten": (ctypes.c_int, [_vp]),
    "csgn_key_create": (ctypes.c_int, [_u64, _vp, ctypes.c_uint32, _vpp]),
    "csgn_key_free": (ctypes.c_int, [_vp]),
    "csgn_decrypt": (ctypes.c_int, [_vp, _vp, ctypes.POINTER(ctypes.c_uint8)]),
    "csgn_decrypt_count": (ctypes.c_int, [_vp, _vp, _u64p]),
    "csgn_decrypt_count_async": (ctypes.c_int, [_vp, _vp, _vp]),
    "csgn_decrypt_product": (ctypes.c_int, [ctypes.POINTER(_vp), ctypes.c_uint32, _vp, ctypes.POINTER(ctypes.c_uint8), _u64p]),
    "csgn_decrypt_deferred": (ctypes.c_int, [_vp, _vp, _vpp]),
    "csgn_result_ready": (ctypes.c_int, [_vp]),
    "csgn_result_wait": (ctypes.c_int, [_vp, _u64p]),
    "csgn_result_free": (ctypes.c_int, [_vp]),
    "csgn_mul_count_async": (ctypes.c_int, [_vp, _vp, _vp, _vpp, _vp]),
    "csgn_mul_decrypt": (ctypes.c_int, [_vp, _vp, _vp, _vpp, ctypes.POINTER(ctypes.c_uint8), _u64p]),
    "csgn_mul_count_batch_async": (ctypes.c_int, [ctypes.POINTER(_vp), ctypes.POINTER(_vp), ctypes.c_uint32, _vp,
                                                  ctypes.POINTER(_vp), _vp]),
    "csgn_mul_decrypt_deferred": (ctypes.c_int, [_vp, _vp, _vp, _vpp, _vpp]),
    "csgn_mul_decrypt_sharded_async": (ctypes.c_int, [_vp, _vp, _vp, _vpp, _vp, ctypes.c_uint32, ctypes.c_uint32, _vp, _vp]),
    "csgn_mul_decrypt_sharded_batch_async": (ctypes.c_int, [ctypes.POINTER(_vp), ctypes.POINTER(_vp), ctypes.c_uint32, _vp,
                                                            ctypes.POINTER(_vp), _vp, ctypes.c_uint32, _vp]),
    "csgn_mul_batch": (ctypes.c_int, [ctypes.POINTER(_vp), ctypes.POINTER(_vp), ctypes.c_uint32, ctypes.POINTER(_vp)]),
    "csgn_mul_into_batch": (ctypes.c_int, [ctypes.POINTER(_vp), ctypes.POINTER(_vp), ctypes.c_uint32, ctypes.POINTER(_vp)]),
    "csgn_decrypt_count_batch_async": (ctypes.c_int, [ctypes.POINTER(_vp), ctypes.c_uint32, _vp, _vp]),
    "csgn_decrypt_batch": (ctypes.c_int, [ctypes.POINTER(_vp), ctypes.c_uint32, _vp, ctypes.POINTER(ctypes.c_uint8), _u64p]),
    "csgn_decrypt_sharded_batch_async": (ctypes.c_int, [ctypes.POINTER(_vp), ctypes.c_uint32, _vp, _vp, ctypes.c_uint32, _vp]),
    "csgn_decrypt_positions": (ctypes.c_int, [_vp, _u64, _vp, ctypes.c_uint32, ctypes.POINTER(ctypes.c_uint8)]),
    "csgn_encrypt_batch": (ctypes.c_int, [_vp, _vp, _u64, _u64, _u64, _vpp]),
    "csgn_seg_mul": (ctypes.c_int, [_vp, _vp, _vp, _vp, _u64, _vp, _vpp]),
    "csgn_seg_concat": (ctypes.c_int, [_vp, _vp, _vp, _vp, _u64, _vp, _vpp]),
    "csgn_seg_mul_sum": (ctypes.c_int, [ctypes.POINTER(_vp), ctypes.POINTER(_vp), ctypes.POINTER(_vp), ctypes.POINTER(_vp),
                                        ctypes.c_uint32, ctypes.POINTER(_vp), ctypes.POINTER(_vp), ctypes.c_uint32, _u64,
                                        _vp, _vpp]),
    "csgn_seg_mul_sum_compact": (ctypes.c_int, [ctypes.POINTER(_vp), ctypes.POINTER(_vp), ctypes.POINTER(_vp),
                                                ctypes.POINTER(_vp), ctypes.c_uint32, ctypes.POINTER(_vp),
                                                ctypes.POINTER(_vp), ctypes.c_uint32, _u64, ctypes.c_uint32, _vp, _vpp]),
    "csgn_seg_cancel": (ctypes.c_int, [_vp, _vp, _u64, _vp, _vpp]),
    "csgn_seg_gather": (ctypes.c_int, [_vp, _vp, _u64, _vp, _u64, _vp, _vpp]),
    "csgn_concat_n": (ctypes.c_int, [ctypes.POINTER(_vp), _u64, _vpp]),
    "csgn_seg_decrypt_count_async": (ctypes.c_int, [_vp, _vp, _u64, _vp, _vp]),
    "csgn_seg_decrypt": (ctypes.c_int, [_vp, _vp, _u64, _vp, _vp, _vp]),
    "csgn_seg_circuit": (ctypes.c_int, [ctypes.POINTER(_vp), ctypes.POINTER(_vp), ctypes.c_uint32, _u64, _vp, _u64,
                                        ctypes.c_uint32, _vp, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_int, _u64,
                                        ctypes.POINTER(_vp), ctypes.POINTER(_vp), _u64p]),
    "csgn_encrypt_uint": (ctypes.c_int, [_vp, _vp, _u64, ctypes.c_uint32, _u64, _u64, ctypes.POINTER(_vp)]),
    "csgn_decrypt_uint_async": (ctypes.c_int, [ctypes.POINTER(_vp), ctypes.POINTER(_vp), ctypes.c_uint32, _u64, _vp, _vp]),
    "csgn_decrypt_uint": (ctypes.c_int, [ctypes.POINTER(_vp), ctypes.POINTER(_vp), ctypes.c_uint32, _u64, _vp, _vp]),
    "csgn_perm_create": (ctypes.c_int, [_u64, _vp, _vpp]),
    "csgn_perm_free": (ctypes.c_int, [_vp]),
    "csgn_permute": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _vpp]),
    "csgn_permute_into": (ctypes.c_int, [_vp, _vp, _vp]),
    "csgn_buf_checksum": (ctypes.c_int, [_vp, _u64p, _u64p, _u64p]),
    "csgn_buf_save": (ctypes.c_int, [_vp, _u64, _u64, ctypes.c_char_p]),
    "csgn_buf_load": (ctypes.c_int, [ctypes.c_char_p, _u64p, _u64p, _vpp]),
    "csgn_buf_save_shard": (ctypes.c_int, [_vp, _u64, _u64, ctypes.c_char_p, ctypes.c_int, ctypes.c_int, _u64]),
    "csgn_buf_load_shard": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_int, ctypes.c_int, _vp, _vp, _vp, _vpp]),
    "csgn_key_positions_save": (ctypes.c_int, [ctypes.c_char_p, _u64, _u64, _vp, _u64]),
    "csgn_key_positions_load": (ctypes.c_int, [ctypes.c_char_p, _vp, _vp, _vp, _u64, _vp]),
    "csgn_perm_entries_save": (ctypes.c_int, [ctypes.c_char_p, _vp, _u64]),
    "csgn_perm_entries_load": (ctypes.c_int, [ctypes.c_char_p, _vp, _u64, _vp]),
    "csgn_shard_range": (ctypes.c_int, [_u64, ctypes.c_int, ctypes.c_int, _u64p, _u64p]),
    "csgn_comm_create": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, _vpp, _vp]),
    "csgn_comm_connect": (ctypes.c_int, [_vp, _vp]),
    "csgn_comm_connect_ptrs": (ctypes.c_int, [_vp, ctypes.POINTER(_vp)]),
    "csgn_comm_connect_dir": (ctypes.c_int, [_vp, _vp, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int]),
    "csgn_comm_mailbox": (_vp, [_vp, ctypes.POINTER(ctypes.c_size_t)]),
    "csgn_comm_free": (ctypes.c_int, [_vp]),
    "csgn_comm_pending": (ctypes.c_uint32, [_vp]),
    "csgn_decrypt_sharded_async": (ctypes.c_int, [_vp, _vp, _vp, ctypes.c_uint32, ctypes.c_uint32, _vp, _vp]),
    "csgn_comm_collect_async": (ctypes.c_int, [_vp, ctypes.c_uint32, ctypes.c_uint32, _vp]),
    "csgn_decrypt_sharded": (ctypes.c_int, [_vp, _vp, _vp, ctypes.POINTER(ctypes.c_uint8), _u64p]),
    "csgn_comm_slot_tag": (None, [_u64, ctypes.POINTER(ctypes.c_uint32), _u64p]),
}

_lib = None


class CsgnError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("csgn error %d: %s" % (code, message))
        self.code = code


def header_path():
    return os.path.join(_build.INCLUDE, "csgn.h")


def declared_symbols():
    """Function names declared in include/csgn.h (parsed, so tests can hold the
    binding table and the shared object to the header)."""
    text = open(header_path()).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(csgn_[a-z_0-9]+)\s*\(", text)))


def load(build_if_missing=True):
    """dlopen libcsgn.so (building it first if sources are newer).  No GPU needed."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.libcsgn_path()
    override = os.environ.get("CSGN_LIBRARY")      # A/B runs of two builds on one GPU box
    if override:
        path, build_if_missing = override, False
    if build_if_missing:
        try:
            _build.build_libcsgn()
        except Exception:
            if not os.path.exists(path):
                raise
    if not os.path.exists(path):
        raise ImportError("CUDA extension %s is missing; build it with `python -m csgn_b200.build` "
                          "(no CPU fallback exists)" % path)
    lib = ctypes.CDLL(path)
    unbound = [name for name in SIGNATURES if override and not hasattr(lib, name)]
    if unbound:                  # an older build under A/B comparison: its newer entry points stay unbound
        warnings.warn("CSGN_LIBRARY=%s lacks %d entry points of include/csgn.h, left unbound: %s"
                      % (path, len(unbound), ", ".join(unbound)))
    for name, (res, args) in SIGNATURES.items():
        if name in unbound:
            continue
        fn = getattr(lib, name)  # AttributeError here = header and library disagree
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise CsgnError(rc, (_lib.csgn_last_error() or b"").decode(errors="replace"))
    return rc
