"""Mirror of the reference's dedup split-archive writer surface, for the hot path only.

Reference (Go, module github.com/pbs-plus/pxar/transfer, call sites in
internal/pxarmount/commit.go):
    writer, err := transfer.NewRemoteDedupSplitArchiveWriter(ctx, session, meta, payload, origPayloadIdx)   :329
    err = writer.WriteEntryReader(entry, reader, size)                                                      :720, :858
    err = writer.Finish()                                                                                   :383
Inside WriteEntryReader the module pulls the reader's bytes, runs the buzhash scan,
cuts, SHA-256s every chunk, asks the session whether the digest is known and uploads
only new chunks.  This mirror keeps the names and the pull-from-a-reader contract but
batches the files: entries are queued and pushed through the GPU engine in one batch on
Flush()/Finish() (SURVEY.md section 8f item 2).  `upload` is a callback (the HTTP/2 upload is out of scope).

Two writers:
  * PayloadStreamWriter -- the LAYOUT-FAITHFUL one and the default for a drop-in: it produces the pxar v2 payload
    stream the production chunker sees (PAYLOAD_START marker, then per file a 16-byte PAYLOAD header + content,
    concatenated: internal/pxarmount/pxarfs.go:408-411), chunks THAT stream through pbsgpu_stream_* with a suggested
    boundary at every file start, returns each entry's payload offset (what the mpxar PAYLOAD_REF stores) and
    supports WriteEntryRef (chunk reuse from the previous .ppxar.didx, commit.go:752, :848-860).
  * DedupWriter -- per-file batching (every file its own stream).  Faster for many small files, but its index does NOT
    describe a ppxar payload stream: use it for dedup statistics / digest computation, not to write .ppxar.didx.
"""
from __future__ import annotations

import io
from dataclasses import dataclass, field
from typing import BinaryIO, Callable

import numpy as np

from ._lib import CHUNK_DTYPE, CHUNK_KNOWN, Cfg
from .engine import DigestSet, Engine


@dataclass
class Entry:
    """The two fields of pxar.Entry the hot path reads (commit.go:710-715)."""
    Path: str
    FileSize: int


@dataclass
class IndexRecord:
    """One dynamic-index entry the writer appends per chunk: (end offset, digest)."""
    path: str
    end_off: int
    digest: bytes
    known: bool


@dataclass
class DedupWriter:
    engine: Engine
    config: Cfg
    known: DigestSet | None = None
    upload: Callable[[bytes, bytes], None] | None = None   # (digest, chunk bytes) for NEW chunks
    # (digest, DataBlob) for NEW chunks: the body of POST /dynamic_chunk (log_cleanup.go:19-31), rendered for all new
    # chunks of a flush by ONE pbsgpu_blob_encode_batch_z call (zstd frame where smaller, CRC-32 from the GPU)
    upload_blob: Callable[[bytes, bytes], None] | None = None
    batch_bytes: int = 1 << 30
    # "rle": frames of RLE / raw blocks (pbsgpu_blob_encode_batch_z); "lz": also Compressed_Blocks from the GPU's match
    # stage (pbsgpu_blob_encode_batch_lz) -- smaller blobs for text-like data at more GPU time per byte
    blob_codec: str = "rle"
    index: list[IndexRecord] = field(default_factory=list)
    # relPath -> XXH3-64 of the file as uploaded: commitWalkState.backedHashes (commit.go:187, :725), computed on the
    # GPU from the same staged bytes instead of through an io.TeeReader on the host
    backed_hashes: dict[str, int] = field(default_factory=dict)
    _pending: list[tuple[Entry, np.ndarray]] = field(default_factory=list)
    _pending_bytes: int = 0
    _finished: bool = False

    def __post_init__(self) -> None:
        if self.blob_codec not in ("rle", "lz"):
            raise ValueError(f"transfer: unknown blob_codec {self.blob_codec!r} (want 'rle' or 'lz')")

    def WriteEntryReader(self, entry: Entry, reader: BinaryIO, size: int) -> None:
        """Pulls exactly `size` bytes from `reader` (error if it yields fewer, like io.ReadFull)."""
        if self._finished:
            raise RuntimeError("transfer: writer already finished")
        data = reader.read(size) if size else b""
        if len(data) != size:
            raise IOError(f"transfer: short read for {entry.Path}: got {len(data)} of {size} bytes (unexpected EOF)")
        self._pending.append((entry, np.frombuffer(data, dtype=np.uint8)))
        self._pending_bytes += size
        if self._pending_bytes >= self.batch_bytes:
            self.Flush()

    def WriteEntry(self, entry: Entry, data: bytes) -> None:
        self.WriteEntryReader(entry, io.BytesIO(data), len(data))

    def Flush(self) -> None:
        if not self._pending:
            return
        entries, arrs = zip(*self._pending)
        buf, offs, lens = self._pack(arrs)
        rec, hashes = self.engine.chunk_digest_batch_xxh3(self.config, buf, offs, lens, self.known)
        for e, h in zip(entries, hashes):
            self.backed_hashes[e.Path] = int(h)
        new_chunks = []                                   # (digest, stream, start, end) of the chunks the server lacks
        starts: dict[int, int] = {}
        for r in rec:
            i = int(r["stream"])
            known = bool(r["flags"] & CHUNK_KNOWN)
            s0, e0 = starts.get(i, 0), int(r["end_off"])
            starts[i] = e0
            self.index.append(IndexRecord(entries[i].Path, e0, bytes(r["digest"]), known))
            if not known:
                new_chunks.append((bytes(r["digest"]), i, s0, e0))
        if self.upload is not None:
            for d, i, s0, e0 in new_chunks:
                self.upload(d, arrs[i][s0:e0].tobytes())
        if self.upload_blob is not None and new_chunks:
            boff = np.array([int(offs[i]) + s0 for _, i, s0, _ in new_chunks], dtype=np.uint64)
            blen = np.array([e0 - s0 for _, _, s0, e0 in new_chunks], dtype=np.uint64)
            encode = self.engine.blob_encode_batch_lz if self.blob_codec == "lz" else self.engine.blob_encode_batch_z
            blobs, _crc = encode(buf, boff, blen)
            for (d, _i, _s, _e), blob in zip(new_chunks, blobs):
                self.upload_blob(d, blob)
        self._pending, self._pending_bytes = [], 0

    @staticmethod
    def _pack(arrs):
        lens = np.array([len(a) for a in arrs], dtype=np.uint64)
        offs = np.zeros(len(arrs), dtype=np.uint64)
        pos = 0
        for i, a in enumerate(arrs):
            offs[i] = pos
            pos += (len(a) + 255) & ~255
        buf = np.zeros(max(pos, 1), dtype=np.uint8)
        for a, o in zip(arrs, offs):
            buf[int(o): int(o) + len(a)] = a
        return buf, offs, lens

    def Finish(self) -> list[IndexRecord]:
        self.Flush()
        self._finished = True
        return self.index


# pxar v2 format constants (upstream pxar crate format/mod.rs; restated, UNVERIFIED against the Go module)
PXAR_PAYLOAD = 0x28147A1B0B7C1A25
PXAR_PAYLOAD_START_MARKER = 0x834C68C2194A4ED2
PXAR_PAYLOAD_TAIL_MARKER = 0x6C72B78B984C81B5


def payload_header(content_len: int) -> bytes:
    """16-byte PAYLOAD header: htype u64 LE, full_size u64 LE (header included) -- pxarfs.go:408-411 skips these 16."""
    return PXAR_PAYLOAD.to_bytes(8, "little") + (16 + content_len).to_bytes(8, "little")


class NotStrictlyGreater(IOError):
    """WriteEntryRef out of order; the message carries the substring the reference matches (commit.go:849)."""


@dataclass
class PayloadStreamWriter:
    """Writes ONE pxar v2 payload stream through the streaming C ABI (see the module docstring)."""
    engine: Engine
    config: Cfg
    known: DigestSet | None = None
    prev_index: tuple[np.ndarray, np.ndarray] | None = None   # (ends u64[], digests u8[n,32]) of the previous .ppxar.didx
    suggest: bool = True             # suggested boundary at every file start (upstream PayloadChunker); False = plain chunker
    index: list[tuple[int, bytes, bool]] = field(default_factory=list)   # (end offset in the NEW stream, digest, known)
    payload_offsets: dict[str, int] = field(default_factory=dict)        # entry path -> offset of its PAYLOAD header
    _stream: object = None
    _seg_base: int = 0               # offset in the new stream at which the current pbsgpu stream starts
    _last_ref: int = -1
    _finished: bool = False

    def __post_init__(self):
        self._open()
        self._raw(PXAR_PAYLOAD_START_MARKER.to_bytes(8, "little") + (16).to_bytes(8, "little"))

    # -- plumbing ---------------------------------------------------------------------------------------------
    def _open(self):
        self._stream = self.engine.stream(self.config, self.known)

    def _raw(self, data: bytes):
        self._stream.write(np.frombuffer(data, dtype=np.uint8))

    @property
    def position(self) -> int:
        return self._seg_base + self._stream.position

    def _drain(self, final: bool):
        rec = self._stream.finish() if final else self._stream.poll(1 << 16)
        for r in rec:
            self.index.append((self._seg_base + int(r["end_off"]), bytes(r["digest"]), bool(r["flags"] & CHUNK_KNOWN)))

    # -- ArchiveWriter surface (commit.go:183) -------------------------------------------------------------------
    def WriteEntryReader(self, entry: Entry, reader: BinaryIO, size: int) -> int:
        """commit.go:720, :858.  Returns the entry's payload offset."""
        if self._finished:
            raise RuntimeError("transfer: writer already finished")
        off = self.position
        if self.suggest and self._stream.position > 0:
            self._stream.suggest(self._stream.position)
        self._raw(payload_header(size))
        left = size
        while left:
            slot = self._stream.reserve()
            want = min(left, len(slot))
            data = reader.read(want)
            if not data:
                self._stream.commit(0)
                raise IOError(f"transfer: short read for {entry.Path}: got {size - left} of {size} bytes (unexpected EOF)")
            slot[: len(data)] = np.frombuffer(data, dtype=np.uint8)
            self._stream.commit(len(data))
            left -= len(data)
        self.payload_offsets[entry.Path] = off
        self._drain(False)
        return off

    def WriteEntryRef(self, entry: Entry, payload_offset: int) -> int:
        """commit.go:752, :848: reuse the previous snapshot's chunks that hold [payload_offset, +16+FileSize) without
        reading the content.  The running chunk is closed, the old chunks are appended to the new index (their bytes
        become part of the new stream, padding included, as in upstream's chunk injection) and the entry's new payload
        offset is returned.  Offsets must ascend; otherwise the error text contains "not strictly greater" and the
        caller re-encodes through WriteEntryReader (commit.go:849-860)."""
        if self.prev_index is None:
            raise IOError("transfer: WriteEntryRef without a previous payload index")
        if payload_offset <= self._last_ref:
            raise NotStrictlyGreater(f"transfer: payload offset {payload_offset} not strictly greater than previous {self._last_ref}")
        ends, digs = self.prev_index
        lo = int(np.searchsorted(ends, payload_offset, side="right"))
        hi = int(np.searchsorted(ends, payload_offset + 16 + entry.FileSize, side="left"))
        if hi >= len(ends):
            raise IOError(f"transfer: payload range of {entry.Path} lies outside the previous index")
        # close the running chunk: the injected chunks start on a chunk boundary of the new stream
        self._drain(True)
        self._seg_base += self._stream.position
        self._stream.close()
        first_start = int(ends[lo - 1]) if lo else 0
        pos = self._seg_base
        for k in range(lo, hi + 1):
            start = int(ends[k - 1]) if k else 0
            pos += int(ends[k]) - start
            self.index.append((pos, bytes(digs[k]), True))
        new_off = self._seg_base + (payload_offset - first_start)
        self._seg_base = pos
        self._last_ref = payload_offset
        self.payload_offsets[entry.Path] = new_off
        self._open()
        return new_off

    def Finish(self) -> list[tuple[int, bytes, bool]]:
        """commit.go:383: tail marker, final short chunk, index complete."""
        if not self._finished:
            self._raw(PXAR_PAYLOAD_TAIL_MARKER.to_bytes(8, "little") + (16).to_bytes(8, "little"))
            self._drain(True)
            self._stream.close()
            self._finished = True
        return self.index

    def didx(self, uuid: bytes = b"\0" * 16, ctime: int = 0) -> bytes:
        """The new .ppxar.didx image (csum on the GPU)."""
        rec = np.zeros(len(self.index), dtype=CHUNK_DTYPE)
        for i, (end, dig, known) in enumerate(self.index):
            rec[i]["end_off"] = end
            rec[i]["digest"] = np.frombuffer(dig, dtype=np.uint8)
            rec[i]["flags"] = CHUNK_KNOWN if known else 0
        return self.engine.didx_build(rec, uuid, ctime)


def NewRemoteDedupSplitArchiveWriter(engine: Engine, config: Cfg, known: DigestSet | None = None,
                                     orig_payload_idx: bytes | None = None, upload=None, upload_blob=None,
                                     blob_codec: str = "rle") -> DedupWriter:
    """commit.go:329.  `orig_payload_idx` = bytes of the previous .ppxar.didx (commit.go:324-328):
    its digests seed the known set, so unchanged chunks are not uploaded again.  `blob_codec` picks the DataBlob
    encoder of `upload_blob` (DedupWriter.blob_codec)."""
    if orig_payload_idx:
        if known is None:
            known = engine.digest_set()
        known.seed_didx(orig_payload_idx)
    return DedupWriter(engine, config, known, upload, upload_blob, blob_codec=blob_codec)


def verifyBackedFileHashes(engine: Engine, open_file: Callable[[str], BinaryIO], hashes: dict[str, int],
                           batch_bytes: int = 1 << 30) -> None:
    """Mirror of verifyBackedFileHashes (reference internal/pxarmount/commit.go:957-976): every backed file is read
    again and its XXH3-64 must equal the value recorded at upload time.  The reference hashes on the host through a
    64 KiB copy buffer, one file at a time; here the files are packed into batches and hashed by ONE
    pbsgpu_xxh3_batch call each.  Errors keep the reference's wording:
    `open backed file "<p>" for verification: ...` and `backed file "<p>" content hash differs`."""
    names: list[str] = []
    arrs: list[np.ndarray] = []
    held = 0

    def flush() -> None:
        nonlocal names, arrs, held
        if not names:
            return
        lens = np.array([len(a) for a in arrs], dtype=np.uint64)
        offs = np.zeros(len(arrs), dtype=np.uint64)
        pos = 0
        for i, a in enumerate(arrs):
            offs[i] = pos
            pos += (len(a) + 255) & ~255
        buf = np.zeros(max(pos, 1), dtype=np.uint8)
        for a, o in zip(arrs, offs):
            buf[int(o): int(o) + len(a)] = a
        got = engine.xxh3_batch(buf, offs, lens)
        for name, h in zip(names, got):
            if int(h) != hashes[name]:
                raise IOError(f'backed file "{name}" content hash differs')
        names, arrs, held = [], [], 0

    for rel in hashes:
        try:
            with open_file(rel) as f:
                data = f.read()
        except OSError as ex:
            raise IOError(f'open backed file "{rel}" for verification: {ex}') from ex
        names.append(rel)
        arrs.append(np.frombuffer(data, dtype=np.uint8))
        held += len(data)
        if held >= batch_bytes:
            flush()
    flush()
