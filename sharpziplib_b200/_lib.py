"""ctypes binding of libb200z.so (include/b200z.h).  The library is the product; this module only loads it.

There is no CPU fallback: if the shared library is missing, or no CUDA device is present when a compute entry point
is called, an exception is raised.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libb200z.so")

OK, E_ARG, E_STATE, E_DATA, E_INTERNAL, E_CUDA, E_UNSUPPORTED, E_NOMEM, E_NEED_INPUT = range(9)
WRAP_RAW, WRAP_ZLIB, WRAP_GZIP, WRAP_RAW_CRC32 = 0, 1, 2, 3
END_FINISH, END_FLUSH_FINISH, END_FLUSH = 0, 1, 2


class SharpZipBaseException(Exception):
    """Mirror of ICSharpCode.SharpZipLib.SharpZipBaseException (Core/Exceptions/SharpZipBaseException.cs)."""


class StreamDecodingException(SharpZipBaseException):
    pass


class B200zUnsupported(NotImplementedError):
    """A call sequence this build does not accelerate (never emulated on the CPU)."""


class B200zCudaError(RuntimeError):
    pass


class InvalidOperationException(RuntimeError):
    pass


def raise_for(rc):
    """status -> the exception class the reference would throw (INTEGRATION.md, SURVEY.md 8b)."""
    if rc == OK:
        return
    msg = lib().b200z_last_error().decode("utf-8", "replace")
    code = rc & 0xFF
    if code == E_ARG:
        raise ValueError(msg)
    if code == E_STATE:
        raise InvalidOperationException(msg)
    if code == E_DATA:
        raise SharpZipBaseException(msg)
    if code == E_UNSUPPORTED:
        raise B200zUnsupported(msg)
    if code == E_CUDA:
        raise B200zCudaError(msg)
    if code == E_NOMEM:
        raise MemoryError(msg)
    if code == E_NEED_INPUT:
        raise SharpZipBaseException("Unexpected EOF")
    raise RuntimeError("b200z status %d: %s" % (rc, msg))


_lib = None

_SIGS = {
    "b200z_last_error": (C.c_char_p, []),
    "b200z_version": (C.c_int, []),
    "b200z_init": (C.c_int, [C.c_int]),
    "b200z_static_tables_size": (C.c_int, []),
    "b200z_static_tables_export": (C.c_int, [C.c_void_p, C.c_int32]),
    "b200z_static_tables_import": (C.c_int, [C.c_void_p, C.c_int32]),
    "b200z_crc32": (C.c_int, [C.c_void_p, C.c_int64, C.POINTER(C.c_uint32)]),
    "b200z_adler32": (C.c_int, [C.c_void_p, C.c_int64, C.POINTER(C.c_uint32)]),
    "b200z_checksum_batch_device": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "b200z_deflate_plan_create": (C.c_int, [C.c_int32, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "b200z_deflate_plan_create_ex": (C.c_int, [C.c_int32, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                               C.POINTER(C.c_void_p)]),
    "b200z_inflate_plan_create": (C.c_int, [C.c_int32, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "b200z_inflate_plan_create_ex": (C.c_int, [C.c_int32, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]),
    "b200z_inflate_plan_set_start_bits": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200z_plan_get_restart_points": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200z_inflate_plan_set_lengths": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200z_plan_get_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "b200z_plan_get_match_table": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200z_plan_data_offset": (C.c_int64, [C.c_void_p, C.c_int32]),
    "b200z_plan_destroy": (C.c_int, [C.c_void_p]),
    "b200z_plan_in_bytes": (C.c_int64, [C.c_void_p]),
    "b200z_plan_out_bytes": (C.c_int64, [C.c_void_p]),
    "b200z_plan_in_offset": (C.c_int64, [C.c_void_p, C.c_int32]),
    "b200z_plan_out_offset": (C.c_int64, [C.c_void_p, C.c_int32]),
    "b200z_plan_out_capacity": (C.c_int64, [C.c_void_p, C.c_int32]),
    "b200z_plan_workspace_bytes": (C.c_int64, [C.c_void_p]),
    "b200z_plan_launches": (C.c_int32, [C.c_void_p]),
    "b200z_plan_set_timing": (C.c_int, [C.c_void_p, C.c_int]),
    "b200z_plan_get_timings": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int32, C.c_void_p, C.c_int32, C.POINTER(C.c_int32)]),
    "b200z_plan_pack": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200z_plan_run": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200z_plan_run_stages": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                        C.c_void_p]),
    "b200z_deflate_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200z_inflate_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200z_release_cached": (C.c_int, []),
    "b200z_device_count": (C.c_int, []),
    "b200z_static_tables_broadcast": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "b200z_aes_derive_keys": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "b200z_aes_state_bytes": (C.c_int64, []),
    "b200z_aes_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_int32,
                                   C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "b200z_aes_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "b200z_aes_transform_create": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_void_p)]),
    "b200z_aes_transform_block": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "b200z_aes_transform_pwd_verifier": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200z_aes_transform_auth_code": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200z_aes_transform_destroy": (C.c_int, [C.c_void_p]),
    "b200z_pkzip_generate_keys": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p]),
    "b200z_pkzip_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]),
    "b200z_pkzip_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]),
    "b200z_partition_by_bytes": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "b200z_deflate_batch_multi": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200z_inflate_batch_multi": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200z_deflate_pipeline_create": (C.c_int, [C.c_int32, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "b200z_inflate_pipeline_create": (C.c_int, [C.c_int32, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "b200z_pipeline_submit": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200z_pipeline_collect": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200z_pipeline_in_flight": (C.c_int32, [C.c_void_p]),
    "b200z_pipeline_destroy": (C.c_int, [C.c_void_p]),
    "b200z_deflate_bound": (C.c_int64, [C.c_int64]),
    "b200z_engine_state_bytes": (C.c_int64, []),
    "b200z_deflater_create": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "b200z_deflater_destroy": (C.c_int, [C.c_void_p]),
    "b200z_deflater_reset": (C.c_int, [C.c_void_p]),
    "b200z_deflater_set_level": (C.c_int, [C.c_void_p, C.c_int]),
    "b200z_deflater_get_level": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "b200z_deflater_set_strategy": (C.c_int, [C.c_void_p, C.c_int]),
    "b200z_deflater_set_dictionary": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32]),
    "b200z_deflater_set_input": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32]),
    "b200z_deflater_flush": (C.c_int, [C.c_void_p]),
    "b200z_deflater_finish": (C.c_int, [C.c_void_p]),
    "b200z_deflater_deflate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(C.c_int32)]),
    "b200z_deflater_needs_input": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "b200z_deflater_is_finished": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "b200z_deflater_total_in": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "b200z_deflater_total_out": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "b200z_deflater_adler": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint32)]),
    "b200z_inflater_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "b200z_inflater_destroy": (C.c_int, [C.c_void_p]),
    "b200z_inflater_reset": (C.c_int, [C.c_void_p]),
    "b200z_inflater_set_dictionary": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32]),
    "b200z_inflater_set_input": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32]),
    "b200z_inflater_inflate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(C.c_int32)]),
    "b200z_inflater_needs_input": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "b200z_inflater_needs_dictionary": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "b200z_inflater_is_finished": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "b200z_inflater_remaining_input": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32)]),
    "b200z_inflater_total_in": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "b200z_inflater_total_out": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "b200z_inflater_adler": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint32)]),
}

EXPORTS = tuple(sorted(_SIGS))

HIST_NONE, HIST_DICTIONARY, HIST_CONTINUE = 0, 1, 2
STAGE_SEARCH, STAGE_ENCODE, STAGE_ALL = 1, 2, 3


class History(C.Structure):
    """b200z_history (include/b200z.h): what a stream's window already holds when its data starts"""
    _fields_ = [("kind", C.c_int32), ("check_seeded", C.c_int32), ("hist_len", C.c_void_p), ("pos_base", C.c_void_p),
                ("bit_base", C.c_void_p), ("hist_mask", C.c_void_p),
                # levels 0-4: SetInput schedule and engine state between segments (NULL = one SetInput, no state)
                ("chunk_count", C.c_void_p), ("chunk_len", C.c_void_p), ("undrained_last", C.c_void_p),
                ("engine_state", C.c_void_p), ("stored_state", C.c_void_p)]


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise ImportError(
                "libb200z.so is not built (run `python -c 'import __graft_entry__ as g; g.build()'` or "
                "sharpziplib_b200/csrc/build.sh); there is no CPU fallback")
        L = C.CDLL(SO_PATH)
        for name, (res, args) in _SIGS.items():
            f = getattr(L, name)
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib


def init(device=0):
    raise_for(lib().b200z_init(device))
