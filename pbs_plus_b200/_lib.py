"""ctypes binding of libpbsgpu.so (C ABI: include/pbsgpu.h).

The product path is the CUDA library.  There is deliberately NO fallback: if the
shared library is missing or no CUDA device is usable, loading / Engine() raises.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "libpbsgpu.so"


class PbsGpuError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"pbsgpu error {code}: {msg}")
        self.code = code


EINVAL, ENOMEM, ERANGE, ECUDA, ENODEV, ESTATE = -22, -12, -34, -5, -19, -77
BATCH_EARLY_INPUT = 1  # pbsgpu_batch_opts.flags


class Cfg(C.Structure):
    _fields_ = [("avg", C.c_uint32), ("min", C.c_uint32), ("max", C.c_uint32), ("mask", C.c_uint32),
                ("break_min", C.c_uint32), ("window", C.c_uint32), ("table", C.c_uint32 * 256)]


class Chunk(C.Structure):
    _fields_ = [("stream", C.c_uint32), ("flags", C.c_uint32), ("end_off", C.c_uint64), ("digest", C.c_uint8 * 32)]


CHUNK_DTYPE = np.dtype([("stream", "<u4"), ("flags", "<u4"), ("end_off", "<u8"), ("digest", "u1", (32,))])
assert CHUNK_DTYPE.itemsize == C.sizeof(Chunk) == 48
CHUNK_KNOWN = 1


class DevInfo(C.Structure):
    _fields_ = [("device", C.c_int32), ("sm_count", C.c_int32), ("cc_major", C.c_int32), ("cc_minor", C.c_int32),
                ("total_mem", C.c_uint64), ("free_mem", C.c_uint64), ("name", C.c_char * 64)]


class Timing(C.Structure):
    _fields_ = [("scan_ms", C.c_float), ("sort_ms", C.c_float), ("resolve_ms", C.c_float), ("sha_ms", C.c_float),
                ("set_ms", C.c_float), ("total_ms", C.c_float), ("scan_t0", C.c_float), ("scan_t1", C.c_float),
                ("sha_t0", C.c_float), ("sha_t1", C.c_float), ("sha_long_ms", C.c_float), ("sha_bulk_ms", C.c_float),
                ("bytes", C.c_uint64), ("chunks", C.c_uint64),
                ("candidates", C.c_uint64), ("scan_launches", C.c_uint32), ("sha_launches", C.c_uint32),
                ("other_launches", C.c_uint32), ("reruns", C.c_uint32)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class BatchOpts(C.Structure):
    """pbsgpu_batch_opts: digest set, suggested boundaries, per-stream XXH3 output."""
    _fields_ = [("size", C.c_uint32), ("flags", C.c_uint32), ("set", C.c_void_p), ("forced_stream", C.c_void_p),
                ("forced_off", C.c_void_p), ("n_forced", C.c_uint64), ("stream_xxh3", C.c_void_p)]


class Corpus(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("file_len", C.c_uint64), ("block_len", C.c_uint64),
                ("run_blocks", C.c_uint32), ("dup_permille", C.c_uint32), ("edit_mode", C.c_uint32),
                ("edit_thresh16", C.c_uint32), ("edit_seed", C.c_uint64)]


# every symbol include/pbsgpu.h declares (tests assert the .so exports all of them)
SYMBOLS = [
    "pbsgpu_version", "pbsgpu_open", "pbsgpu_close", "pbsgpu_strerror", "pbsgpu_device_info",
    "pbsgpu_set_profiling", "pbsgpu_partition_info", "pbsgpu_scan_partition_sms", "pbsgpu_set_kernel_variant", "pbsgpu_config", "pbsgpu_config_kib",
    "pbsgpu_default_table", "pbsgpu_chunk_digest_batch", "pbsgpu_batch_submit", "pbsgpu_batch_wait",
    "pbsgpu_chunk_digest_batch_ex", "pbsgpu_batch_submit_ex", "pbsgpu_batch_free", "pbsgpu_batch_wait_input", "pbsgpu_batch_input_done",
    "pbsgpu_scan_batch", "pbsgpu_sha256_batch", "pbsgpu_stream_open", "pbsgpu_stream_write",
    "pbsgpu_stream_poll", "pbsgpu_stream_finish", "pbsgpu_stream_close", "pbsgpu_stream_reserve", "pbsgpu_stream_commit",
    "pbsgpu_stream_slot_bytes", "pbsgpu_stream_suggest", "pbsgpu_stream_position", "pbsgpu_set_create",
    "pbsgpu_set_destroy", "pbsgpu_set_insert", "pbsgpu_set_probe", "pbsgpu_set_count", "pbsgpu_set_seed_didx",
    "pbsgpu_set_allgather", "pbsgpu_nccl_unique_id", "pbsgpu_nccl_comm_create", "pbsgpu_nccl_comm_destroy",
    "pbsgpu_didx_size", "pbsgpu_didx_build", "pbsgpu_didx_parse", "pbsgpu_crc32_batch", "pbsgpu_blob_header",
    "pbsgpu_blob_size", "pbsgpu_blob_encode_batch", "pbsgpu_blob_encode_batch_z", "pbsgpu_blob_encode_batch_lz",
    "pbsgpu_xxh3_batch", "pbsgpu_chunk_digest_batch_xxh3",
    "pbsgpu_host_alloc", "pbsgpu_host_free", "pbsgpu_corpus_fill",
]

_lib = None


def lib() -> C.CDLL:
    """Load libpbsgpu.so (fails loudly when the CUDA extension has not been built)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} not found: the CUDA extension is the product and there is no fallback. "
            "Build it with `python -m pbs_plus_b200.build` (or __graft_entry__.build()).")
    L = C.CDLL(str(LIB_PATH))
    vp, u32p, u64p = C.c_void_p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)
    L.pbsgpu_version.restype = C.c_int
    L.pbsgpu_open.argtypes = [C.c_int, C.POINTER(vp)]
    L.pbsgpu_close.argtypes = [vp]
    L.pbsgpu_close.restype = None
    L.pbsgpu_strerror.argtypes = [vp]
    L.pbsgpu_strerror.restype = C.c_char_p
    L.pbsgpu_device_info.argtypes = [vp, C.POINTER(DevInfo)]
    L.pbsgpu_set_profiling.argtypes = [vp, C.c_int]
    L.pbsgpu_partition_info.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.pbsgpu_scan_partition_sms.argtypes = [vp]
    L.pbsgpu_set_kernel_variant.argtypes = [vp, C.c_int]
    L.pbsgpu_config.argtypes = [C.c_uint32, u32p, C.POINTER(Cfg)]
    L.pbsgpu_config_kib.argtypes = [C.c_uint32, u32p, C.POINTER(Cfg)]
    L.pbsgpu_default_table.restype = u32p
    L.pbsgpu_chunk_digest_batch.argtypes = [vp, C.POINTER(Cfg), vp, vp, vp, C.c_uint32, vp, vp, C.c_uint64, u64p]
    L.pbsgpu_batch_submit.argtypes = [vp, C.POINTER(Cfg), vp, vp, vp, C.c_uint32, C.POINTER(vp)]
    L.pbsgpu_batch_wait.argtypes = [vp, vp, C.c_uint64, u64p, C.POINTER(Timing)]
    L.pbsgpu_chunk_digest_batch_ex.argtypes = [vp, C.POINTER(Cfg), vp, vp, vp, C.c_uint32, C.POINTER(BatchOpts), vp, C.c_uint64, u64p]
    L.pbsgpu_batch_submit_ex.argtypes = [vp, C.POINTER(Cfg), vp, vp, vp, C.c_uint32, C.POINTER(BatchOpts), C.POINTER(vp)]
    L.pbsgpu_batch_free.argtypes = [vp]
    L.pbsgpu_batch_wait_input.argtypes = [vp]
    L.pbsgpu_batch_input_done.argtypes = [vp]
    L.pbsgpu_batch_free.restype = None
    L.pbsgpu_scan_batch.argtypes = [vp, C.POINTER(Cfg), vp, vp, vp, C.c_uint32, vp, C.c_uint64, vp, u64p]
    L.pbsgpu_sha256_batch.argtypes = [vp, vp, vp, vp, C.c_uint32, vp]
    L.pbsgpu_stream_open.argtypes = [vp, C.POINTER(Cfg), vp, C.POINTER(vp)]
    L.pbsgpu_stream_write.argtypes = [vp, vp, C.c_uint64]
    L.pbsgpu_stream_poll.argtypes = [vp, vp, C.c_uint64, u64p]
    L.pbsgpu_stream_finish.argtypes = [vp]
    L.pbsgpu_stream_close.argtypes = [vp]
    L.pbsgpu_stream_close.restype = None
    L.pbsgpu_stream_reserve.argtypes = [vp, C.POINTER(vp)]
    L.pbsgpu_stream_commit.argtypes = [vp, C.c_uint64]
    L.pbsgpu_stream_slot_bytes.argtypes = [vp]
    L.pbsgpu_stream_slot_bytes.restype = C.c_uint64
    L.pbsgpu_stream_suggest.argtypes = [vp, C.c_uint64]
    L.pbsgpu_stream_position.argtypes = [vp]
    L.pbsgpu_stream_position.restype = C.c_uint64
    L.pbsgpu_set_allgather.argtypes = [vp, vp, vp, C.c_uint64, vp]
    L.pbsgpu_nccl_unique_id.argtypes = [vp]
    L.pbsgpu_nccl_comm_create.argtypes = [vp, vp, C.c_int, C.c_int, C.POINTER(vp)]
    L.pbsgpu_nccl_comm_destroy.argtypes = [vp]
    L.pbsgpu_nccl_comm_destroy.restype = None
    L.pbsgpu_blob_size.argtypes = [C.c_uint64]
    L.pbsgpu_blob_size.restype = C.c_uint64
    L.pbsgpu_blob_encode_batch.argtypes = [vp, vp, vp, vp, C.c_uint32, vp, vp, vp]
    L.pbsgpu_blob_encode_batch_z.argtypes = [vp, vp, vp, vp, C.c_uint32, vp, vp, vp, vp]
    L.pbsgpu_blob_encode_batch_lz.argtypes = [vp, vp, vp, vp, C.c_uint32, vp, vp, vp, vp]
    L.pbsgpu_set_create.argtypes = [vp, C.c_uint64, C.POINTER(vp)]
    L.pbsgpu_set_destroy.argtypes = [vp]
    L.pbsgpu_set_destroy.restype = None
    L.pbsgpu_set_insert.argtypes = [vp, vp, C.c_uint64, vp]
    L.pbsgpu_set_probe.argtypes = [vp, vp, C.c_uint64, vp]
    L.pbsgpu_set_count.argtypes = [vp, u64p]
    L.pbsgpu_set_seed_didx.argtypes = [vp, vp, C.c_uint64, u64p]
    L.pbsgpu_didx_size.argtypes = [C.c_uint64]
    L.pbsgpu_didx_size.restype = C.c_uint64
    L.pbsgpu_didx_build.argtypes = [vp, vp, C.c_uint64, vp, C.c_int64, vp, C.c_uint64]
    L.pbsgpu_didx_parse.argtypes = [vp, vp, C.c_uint64, vp, vp, C.c_uint64, u64p, C.c_int]
    L.pbsgpu_crc32_batch.argtypes = [vp, vp, vp, vp, C.c_uint32, vp]
    L.pbsgpu_xxh3_batch.argtypes = [vp, vp, vp, vp, C.c_uint32, vp]
    L.pbsgpu_chunk_digest_batch_xxh3.argtypes = [vp, C.POINTER(Cfg), vp, vp, vp, C.c_uint32, vp, vp, C.c_uint64, u64p, vp]
    L.pbsgpu_blob_header.argtypes = [C.c_uint32, vp]
    L.pbsgpu_blob_header.restype = None
    L.pbsgpu_host_alloc.argtypes = [vp, C.c_uint64]
    L.pbsgpu_host_alloc.restype = vp
    L.pbsgpu_host_free.argtypes = [vp, vp]
    L.pbsgpu_host_free.restype = None
    L.pbsgpu_corpus_fill.argtypes = [vp, C.POINTER(Corpus), C.c_uint64, C.c_uint32, vp, C.c_uint64]
    _lib = L
    return L
