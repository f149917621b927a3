"""Host-side front end of the B200 chunk + digest + probe engine.

Thin, allocation-free wrappers over the C ABI (include/pbsgpu.h).  Device memory
comes from the caller (e.g. a torch CUDA tensor -- torch is plumbing only) or the
library stages host memory itself.  No CPU fallback: everything below runs the
sm_100a kernels in pbs_plus_b200/csrc/.
"""
from __future__ import annotations

import ctypes as C
from typing import Iterable, Sequence

import numpy as np

from . import _lib
from ._lib import CHUNK_DTYPE, CHUNK_KNOWN, BatchOpts, Cfg, Corpus, DevInfo, PbsGpuError, Timing


def _ptr(x) -> int:
    """Raw address of a torch tensor / numpy array / int."""
    if isinstance(x, int):
        return x
    if hasattr(x, "data_ptr"):
        return int(x.data_ptr())
    if isinstance(x, np.ndarray):
        return int(x.ctypes.data)
    if isinstance(x, (bytes, bytearray, memoryview)):
        return int(np.frombuffer(x, dtype=np.uint8).ctypes.data)
    raise TypeError(f"cannot take the address of {type(x)}")


def make_config(avg_bytes: int, table: np.ndarray | None = None) -> Cfg:
    """Chunker parameters; replaces buzhash.NewConfig (reference commit.go:302-305). avg in BYTES."""
    cfg = Cfg()
    tp = None
    if table is not None:
        table = np.ascontiguousarray(table, dtype=np.uint32)
        if table.shape != (256,):
            raise ValueError("table must hold 256 u32 entries")
        tp = table.ctypes.data_as(C.POINTER(C.c_uint32))
    rc = _lib.lib().pbsgpu_config(int(avg_bytes), tp, C.byref(cfg))
    if rc:
        raise PbsGpuError(rc, f"invalid average chunk size {avg_bytes} (power of two in [256, 2^29] required)")
    return cfg


def default_table() -> np.ndarray:
    return np.ctypeslib.as_array(_lib.lib().pbsgpu_default_table(), shape=(256,)).copy()


class Engine:
    """One context on one GPU (pbsgpu_open).  Raises if the device or the .so is missing."""

    def __init__(self, device: int = 0, profiling: bool = False):
        self._L = _lib.lib()
        h = C.c_void_p()
        rc = self._L.pbsgpu_open(device, C.byref(h))
        if rc:
            raise PbsGpuError(rc, "pbsgpu_open failed: no usable CUDA device (there is no CPU fallback)")
        self._h = h
        self.device = device
        if profiling:
            self.set_profiling(True)

    # -- plumbing ------------------------------------------------------------------
    def _ck(self, rc: int):
        if rc:
            raise PbsGpuError(rc, (self._L.pbsgpu_strerror(self._h) or b"").decode())

    def close(self):
        if getattr(self, "_h", None):
            self._L.pbsgpu_close(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def device_info(self) -> dict:
        d = DevInfo()
        self._ck(self._L.pbsgpu_device_info(self._h, C.byref(d)))
        return {"device": d.device, "sm_count": d.sm_count, "cc": (d.cc_major, d.cc_minor),
                "total_mem": d.total_mem, "free_mem": d.free_mem, "name": d.name.decode()}

    def partition_info(self) -> tuple[int, int]:
        """(SMs reserved for long-chunk kernels, SMs for the rest); (0, 0) if not partitioned."""
        a, b = C.c_int(), C.c_int()
        self._ck(self._L.pbsgpu_partition_info(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def scan_partition_sms(self) -> int:
        """SMs reserved for the front halves (K1 scan / sort / K2 resolve); 0 = shared with the bulk partition."""
        return int(self._L.pbsgpu_scan_partition_sms(self._h))

    def set_profiling(self, on: bool):
        self._ck(self._L.pbsgpu_set_profiling(self._h, 1 if on else 0))

    def set_kernel_variant(self, variant: int):
        """0 = tuned kernels, 1 = simple cross-check kernels (identical results)."""
        self._ck(self._L.pbsgpu_set_kernel_variant(self._h, variant))

    # -- a2+a3(+a4): batch ----------------------------------------------------------
    @staticmethod
    def _offlen(off: Sequence[int], length: Sequence[int]):
        o = np.ascontiguousarray(off, dtype=np.uint64)
        l = np.ascontiguousarray(length, dtype=np.uint64)
        if o.shape != l.shape or o.ndim != 1:
            raise ValueError("off/len must be 1-D and of equal length")
        return o, l

    @staticmethod
    def _chunk_cap(cfg: Cfg, l: np.ndarray) -> int:
        m = max(int(cfg.min), 65)
        return int((l // np.uint64(m)).sum()) + len(l) + 1

    @staticmethod
    def _opts(digest_set, forced, xxh3=None):
        """pbsgpu_batch_opts; `forced` = (stream u32[], offset u64[]) suggested boundaries sorted by (stream, offset)."""
        o = BatchOpts()
        o.size = C.sizeof(BatchOpts)
        o.set = digest_set._h if digest_set is not None else None
        keep = []
        if forced is not None:
            fs = np.ascontiguousarray(forced[0], dtype=np.uint32)
            fo = np.ascontiguousarray(forced[1], dtype=np.uint64)
            if fs.shape != fo.shape or fs.ndim != 1:
                raise ValueError("forced = (stream[], offset[]) of equal length")
            o.forced_stream, o.forced_off, o.n_forced = fs.ctypes.data, fo.ctypes.data, len(fs)
            keep += [fs, fo]
        if xxh3 is not None:
            o.stream_xxh3 = xxh3.ctypes.data
        return o, keep

    def chunk_digest_batch(self, cfg: Cfg, base, off, length, digest_set: "DigestSet | None" = None,
                           forced=None) -> np.ndarray:
        """stream -> chunks -> digests for n streams; `base` device (tensor/int) or host (numpy).
        Replaces n calls of writer.WriteEntryReader (reference commit.go:720).  `forced` = optional suggested
        boundaries (stream[], offset[]): file starts of a pxar payload stream (pxarfs.go:408-411)."""
        o, l = self._offlen(off, length)
        cap = self._chunk_cap(cfg, l) + (len(forced[0]) if forced is not None else 0)
        out = np.zeros(cap, dtype=CHUNK_DTYPE)
        n_out = C.c_uint64()
        keep = base  # keep the buffer alive for the duration of the call
        opts, _k = self._opts(digest_set, forced)
        self._ck(self._L.pbsgpu_chunk_digest_batch_ex(
            self._h, C.byref(cfg), _ptr(keep), o.ctypes.data, l.ctypes.data, len(o), C.byref(opts), out.ctypes.data, cap,
            C.byref(n_out)))
        return out[: n_out.value]

    def chunk_digest_batch_xxh3(self, cfg: Cfg, base, off, length, digest_set: "DigestSet | None" = None):
        """chunk_digest_batch plus the XXH3-64 of every stream from the same staged bytes (f2: the per-file
        hash of emitBackedFile, reference commit.go:717-725).  Returns (chunks, xxh3[n] uint64)."""
        o, l = self._offlen(off, length)
        cap = self._chunk_cap(cfg, l)
        out = np.zeros(cap, dtype=CHUNK_DTYPE)
        hashes = np.zeros(len(o), dtype=np.uint64)
        n_out = C.c_uint64()
        keep = base
        self._ck(self._L.pbsgpu_chunk_digest_batch_xxh3(
            self._h, C.byref(cfg), _ptr(keep), o.ctypes.data, l.ctypes.data, len(o),
            digest_set._h if digest_set is not None else None, out.ctypes.data, cap, C.byref(n_out), hashes.ctypes.data))
        return out[: n_out.value], hashes

    def chunk_digest_streams(self, cfg: Cfg, streams: Iterable[np.ndarray], digest_set=None) -> np.ndarray:
        """Convenience for host streams that are separate arrays: packs them and calls the batch ABI."""
        arrs = [np.ascontiguousarray(s, dtype=np.uint8) for s in streams]
        lens = np.array([len(a) for a in arrs], dtype=np.uint64)
        offs = np.zeros(len(arrs), dtype=np.uint64)
        pos = 0
        for i, a in enumerate(arrs):
            offs[i] = pos
            pos += (len(a) + 255) & ~255
        buf = np.zeros(max(pos, 1), dtype=np.uint8)
        for a, o in zip(arrs, offs):
            buf[int(o): int(o) + len(a)] = a
        return self.chunk_digest_batch(cfg, buf, offs, lens, digest_set)

    def submit(self, cfg: Cfg, base_dev, off, length, digest_set: "DigestSet | None" = None, forced=None,
               early_input: bool = False) -> "Job":
        """Asynchronous form; with `digest_set` the probe + insert runs as kernels on the job's stream (jobs sharing a
        set are ordered in submission order) and the KNOWN flags come back with the records.  `early_input`
        (PBSGPU_BATCH_EARLY_INPUT): the long chunks are copied aside so that Job.wait_input() gives the buffer back
        long before the records are ready."""
        o, l = self._offlen(off, length)
        h = C.c_void_p()
        opts, _k = self._opts(digest_set, forced)
        if early_input:
            opts.flags |= _lib.BATCH_EARLY_INPUT
        self._ck(self._L.pbsgpu_batch_submit_ex(self._h, C.byref(cfg), _ptr(base_dev), o.ctypes.data, l.ctypes.data,
                                                len(o), C.byref(opts), C.byref(h)))
        return Job(self, h, self._chunk_cap(cfg, l) + (len(forced[0]) if forced is not None else 0), base_dev)

    def scan_batch(self, cfg: Cfg, base_dev, off, length):
        """Boundaries only (a2).  Returns (ends, stream_first)."""
        o, l = self._offlen(off, length)
        cap = self._chunk_cap(cfg, l)
        ends = np.zeros(cap, dtype=np.uint64)
        first = np.zeros(len(o) + 1, dtype=np.uint64)
        n_out = C.c_uint64()
        self._ck(self._L.pbsgpu_scan_batch(self._h, C.byref(cfg), _ptr(base_dev), o.ctypes.data, l.ctypes.data,
                                           len(o), ends.ctypes.data, cap, first.ctypes.data, C.byref(n_out)))
        return ends[: n_out.value], first

    def sha256_batch(self, base, off, length) -> np.ndarray:
        """SHA-256 of n byte ranges (a3); returns (n, 32) uint8."""
        o, l = self._offlen(off, length)
        out = np.zeros((len(o), 32), dtype=np.uint8)
        self._ck(self._L.pbsgpu_sha256_batch(self._h, _ptr(base), o.ctypes.data, l.ctypes.data, len(o),
                                             out.ctypes.data))
        return out

    # -- f2: per-file content hash of the commit walk ---------------------------------------------
    def xxh3_batch(self, base, off, length) -> np.ndarray:
        """XXH3-64 (seed 0) of n byte ranges (host or device base) on the GPU; uint64[n]."""
        o, l = self._offlen(off, length)
        out = np.zeros(len(o), dtype=np.uint64)
        self._ck(self._L.pbsgpu_xxh3_batch(self._h, _ptr(base), o.ctypes.data, l.ctypes.data, len(o), out.ctypes.data))
        return out

    # -- f3: DataBlob checksums --------------------------------------------------------------
    def crc32_batch(self, base, off, length) -> np.ndarray:
        """zlib-compatible CRC-32 of n byte ranges (host or device base) on the GPU."""
        o, l = self._offlen(off, length)
        out = np.zeros(len(o), dtype=np.uint32)
        self._ck(self._L.pbsgpu_crc32_batch(self._h, _ptr(base), o.ctypes.data, l.ctypes.data, len(o), out.ctypes.data))
        return out

    def blob_encode_batch(self, base, off, length):
        """Complete uncompressed DataBlobs (magic | crc32 | payload) of n ranges -> (bytes buffer, blob_off[n+1], crc[n])."""
        o, l = self._offlen(off, length)
        sizes = l + np.uint64(12)
        boff = np.zeros(len(o) + 1, dtype=np.uint64)
        np.cumsum(sizes, out=boff[1:])
        out = np.zeros(int(boff[-1]), dtype=np.uint8)
        crc = np.zeros(len(o), dtype=np.uint32)
        self._ck(self._L.pbsgpu_blob_encode_batch(self._h, _ptr(base), o.ctypes.data, l.ctypes.data, len(o),
                                                  out.ctypes.data if len(out) else None, boff.ctypes.data, crc.ctypes.data))
        return out, boff, crc

    def blob_encode_batch_z(self, base, off, length):
        """DataBlobs with a zstd payload where that is smaller (RLE / raw block frames, pbsgpu_blob_encode_batch_z)
        -> list of n `bytes` blobs, crc[n]."""
        return self._blob_encode_zstd(self._L.pbsgpu_blob_encode_batch_z, base, off, length)

    def blob_encode_batch_lz(self, base, off, length):
        """blob_encode_batch_z whose frames also hold Compressed_Blocks from the GPU's greedy LZ parse where those are
        smaller (pbsgpu_blob_encode_batch_lz) -> list of n `bytes` blobs, crc[n]."""
        return self._blob_encode_zstd(self._L.pbsgpu_blob_encode_batch_lz, base, off, length)

    def _blob_encode_zstd(self, fn, base, off, length):
        o, l = self._offlen(off, length)
        sizes = l + np.uint64(12)
        boff = np.zeros(len(o) + 1, dtype=np.uint64)
        np.cumsum(sizes, out=boff[1:])
        out = np.zeros(max(1, int(boff[-1])), dtype=np.uint8)
        blen = np.zeros(len(o), dtype=np.uint64)
        crc = np.zeros(len(o), dtype=np.uint32)
        self._ck(fn(self._h, _ptr(base), o.ctypes.data, l.ctypes.data, len(o), out.ctypes.data, boff.ctypes.data,
                    blen.ctypes.data, crc.ctypes.data))
        return [out[int(boff[i]): int(boff[i]) + int(blen[i])].tobytes() for i in range(len(o))], crc

    def blob_header(self, crc: int) -> bytes:
        out = np.zeros(12, dtype=np.uint8)
        self._L.pbsgpu_blob_header(int(crc), out.ctypes.data)
        return out.tobytes()

    # -- f1: dynamic index images ---------------------------------------------------------
    def didx_build(self, chunks: np.ndarray, uuid: bytes = b"\0" * 16, ctime: int = 0) -> bytes:
        """Dynamic-index (.didx) image of chunk records in (stream, offset) order; offsets cumulative."""
        rec = np.ascontiguousarray(chunks, dtype=CHUNK_DTYPE)
        size = int(self._L.pbsgpu_didx_size(len(rec)))
        out = np.zeros(size, dtype=np.uint8)
        u = np.frombuffer(bytes(uuid).ljust(16, b"\0")[:16], dtype=np.uint8)
        self._ck(self._L.pbsgpu_didx_build(self._h, rec.ctypes.data if len(rec) else None, len(rec), u.ctypes.data,
                                           int(ctime), out.ctypes.data, size))
        return out.tobytes()

    def didx_parse(self, image: bytes, verify: bool = True):
        """-> (ends u64[n], digests u8[n,32]); verify recomputes the index checksum on the GPU."""
        a = np.frombuffer(image, dtype=np.uint8)
        n = C.c_uint64()
        self._ck(self._L.pbsgpu_didx_parse(self._h, a.ctypes.data, len(a), None, None, 0, C.byref(n), 0))
        ends = np.zeros(n.value, dtype=np.uint64)
        dig = np.zeros((n.value, 32), dtype=np.uint8)
        self._ck(self._L.pbsgpu_didx_parse(self._h, a.ctypes.data, len(a), ends.ctypes.data, dig.ctypes.data, n.value,
                                           C.byref(n), 1 if verify else 0))
        return ends, dig

    # -- misc ---------------------------------------------------------------------------
    def digest_set(self, capacity_hint: int = 1 << 16) -> "DigestSet":
        return DigestSet(self, capacity_hint)

    def stream(self, cfg: Cfg, digest_set: "DigestSet | None" = None) -> "Stream":
        return Stream(self, cfg, digest_set)

    def host_alloc(self, nbytes: int) -> np.ndarray:
        """Pinned host staging owned by the library (what the Go side would fill)."""
        p = self._L.pbsgpu_host_alloc(self._h, nbytes)
        if not p:
            raise PbsGpuError(_lib.ENOMEM, f"pinned allocation of {nbytes} bytes failed")
        arr = np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(p))
        arr = arr.view(_PinnedArray)
        arr._engine, arr._addr = self, p
        return arr

    def host_free(self, arr):
        addr = getattr(arr, "_addr", None)
        if addr:
            self._L.pbsgpu_host_free(self._h, addr)
            arr._addr = None

    def corpus_fill(self, corpus: Corpus, first_file: int, n_files: int, dst_dev, stride: int):
        self._ck(self._L.pbsgpu_corpus_fill(self._h, C.byref(corpus), first_file, n_files, _ptr(dst_dev), stride))


class _PinnedArray(np.ndarray):
    _engine = None
    _addr = None


class Job:
    """An in-flight batch (pbsgpu_batch_submit); several may overlap on the GPU."""

    def __init__(self, eng: Engine, h, cap: int, keepalive):
        self._eng, self._h, self._cap, self._keep = eng, h, cap, keepalive

    def wait(self):
        out = np.zeros(self._cap, dtype=CHUNK_DTYPE)
        n_out = C.c_uint64()
        t = Timing()
        h = self._h
        rc = self._eng._L.pbsgpu_batch_wait(h, out.ctypes.data, self._cap, C.byref(n_out), C.byref(t))
        if rc == _lib.ERANGE:                       # the job stays valid: retry with the reported capacity
            self._cap = int(n_out.value)
            out = np.zeros(self._cap, dtype=CHUNK_DTYPE)
            rc = self._eng._L.pbsgpu_batch_wait(h, out.ctypes.data, self._cap, C.byref(n_out), C.byref(t))
        self._h = None
        self._eng._ck(rc)
        self._keep = None
        return out[: n_out.value], t.as_dict()

    def wait_input(self):
        """Blocks until the device no longer reads the input buffer (pbsgpu_batch_wait_input); the job stays in flight."""
        self._eng._ck(self._eng._L.pbsgpu_batch_wait_input(self._h))
        self._keep = None

    def input_done(self) -> bool:
        """Non-blocking form of wait_input."""
        rc = self._eng._L.pbsgpu_batch_input_done(self._h)
        if rc < 0:
            self._eng._ck(rc)
        return rc == 1

    def free(self):
        """Abandon the job (pbsgpu_batch_free)."""
        if self._h is not None:
            self._eng._L.pbsgpu_batch_free(self._h)
            self._h, self._keep = None, None


class DigestSet:
    """Known-digest set on the device (reference: dedup seed, commit.go:286-294, :324-329)."""

    def __init__(self, eng: Engine, capacity_hint: int):
        self._eng = eng
        h = C.c_void_p()
        eng._ck(eng._L.pbsgpu_set_create(eng._h, capacity_hint, C.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None) and self._eng._h:
            self._eng._L.pbsgpu_set_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __len__(self):
        c = C.c_uint64()
        self._eng._ck(self._eng._L.pbsgpu_set_count(self._h, C.byref(c)))
        return int(c.value)

    def _run(self, fn, digests):
        d = np.ascontiguousarray(digests, dtype=np.uint8).reshape(-1, 32)
        hit = np.zeros(len(d), dtype=np.uint8)
        self._eng._ck(fn(self._h, d.ctypes.data if len(d) else None, len(d), hit.ctypes.data if len(d) else None))
        return hit

    def insert(self, digests) -> np.ndarray:
        """Insert; returns hit[i] = 1 if digest i was already known (before or earlier in this call)."""
        return self._run(self._eng._L.pbsgpu_set_insert, digests)

    def probe(self, digests) -> np.ndarray:
        return self._run(self._eng._L.pbsgpu_set_probe, digests)

    def allgather(self, comm: "NcclComm", digests) -> np.ndarray:
        """The ONE multi-GPU exchange step (pbsgpu_set_allgather): every rank contributes its digests, every replica
        inserts all of them in global (rank, index) order; returns this rank's flags."""
        d = np.ascontiguousarray(digests, dtype=np.uint8).reshape(-1, 32)
        hit = np.zeros(len(d), dtype=np.uint8)
        self._eng._ck(self._eng._L.pbsgpu_set_allgather(self._h, comm._h, d.ctypes.data if len(d) else None, len(d),
                                                         hit.ctypes.data if len(d) else None))
        return hit

    def seed_didx(self, image: bytes) -> int:
        a = np.frombuffer(image, dtype=np.uint8)
        n = C.c_uint64()
        self._eng._ck(self._eng._L.pbsgpu_set_seed_didx(self._h, a.ctypes.data, len(a), C.byref(n)))
        return int(n.value)


class NcclComm:
    """An ncclComm_t created through the C ABI's helpers (no torch): rank 0 makes the unique id, every rank passes
    the same 128 bytes (distributed by whatever channel the ranks share) to pbsgpu_nccl_comm_create."""

    def __init__(self, eng: Engine, unique_id: bytes, nranks: int, rank: int):
        self._eng = eng
        ida = np.frombuffer(bytes(unique_id), dtype=np.uint8)
        if len(ida) != 128:
            raise ValueError("NCCL unique id is 128 bytes")
        h = C.c_void_p()
        eng._ck(eng._L.pbsgpu_nccl_comm_create(eng._h, ida.ctypes.data, nranks, rank, C.byref(h)))
        self._h = h

    @staticmethod
    def unique_id() -> bytes:
        out = np.zeros(128, dtype=np.uint8)
        rc = _lib.lib().pbsgpu_nccl_unique_id(out.ctypes.data)
        if rc:
            raise PbsGpuError(rc, "NCCL unavailable (libnccl.so.2 not loadable; set PBSGPU_NCCL_LIB)")
        return out.tobytes()

    def close(self):
        if getattr(self, "_h", None):
            self._eng._L.pbsgpu_nccl_comm_destroy(self._h)
            self._h = None


class Stream:
    """Streaming form: one io.Reader-like byte stream, state carried across writes."""

    def __init__(self, eng: Engine, cfg: Cfg, digest_set: DigestSet | None):
        self._eng = eng
        h = C.c_void_p()
        eng._ck(eng._L.pbsgpu_stream_open(eng._h, C.byref(cfg), digest_set._h if digest_set else None, C.byref(h)))
        self._h = h

    def write(self, data):
        a = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else np.ascontiguousarray(data)
        self._eng._ck(self._eng._L.pbsgpu_stream_write(self._h, a.ctypes.data if len(a) else None, len(a)))

    def suggest(self, offset: int):
        """Suggested boundary (a file's PAYLOAD header starts here) -- pbsgpu_stream_suggest."""
        self._eng._ck(self._eng._L.pbsgpu_stream_suggest(self._h, int(offset)))

    @property
    def position(self) -> int:
        return int(self._eng._L.pbsgpu_stream_position(self._h))

    def reserve(self) -> np.ndarray:
        """A pinned staging slot owned by the stream; fill a prefix and call commit(n)."""
        p = C.c_void_p()
        self._eng._ck(self._eng._L.pbsgpu_stream_reserve(self._h, C.byref(p)))
        n = int(self._eng._L.pbsgpu_stream_slot_bytes(self._h))
        return np.ctypeslib.as_array((C.c_uint8 * n).from_address(p.value))

    def commit(self, n: int):
        self._eng._ck(self._eng._L.pbsgpu_stream_commit(self._h, int(n)))

    def poll(self, cap: int = 4096) -> np.ndarray:
        out = np.zeros(cap, dtype=CHUNK_DTYPE)
        n = C.c_uint64()
        self._eng._ck(self._eng._L.pbsgpu_stream_poll(self._h, out.ctypes.data, cap, C.byref(n)))
        return out[: n.value]

    def finish(self) -> np.ndarray:
        self._eng._ck(self._eng._L.pbsgpu_stream_finish(self._h))
        parts = []
        while True:
            p = self.poll()
            if len(p) == 0:
                break
            parts.append(p)
        return np.concatenate(parts) if parts else np.zeros(0, dtype=CHUNK_DTYPE)

    def close(self):
        if getattr(self, "_h", None) and self._eng._h:
            self._eng._L.pbsgpu_stream_close(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def corpus(seed: int, file_len: int, block_len: int = 4 << 20, run_blocks: int = 8, dup_permille: int = 0,
           edit_mode: int = 0, edit_thresh16: int = 655, edit_seed: int = 5) -> Corpus:
    return Corpus(seed, file_len, block_len, run_blocks, dup_permille, edit_mode, edit_thresh16, edit_seed)
