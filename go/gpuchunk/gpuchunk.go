//go:build gpu && cgo

// Package gpuchunk is the cgo shim a pbs-plus maintainer adds to call libpbsgpu.so
// (include/pbsgpu.h) from the Go host code.  It is the reference-side binding for the
// ONE hot path this repository accelerates: buzhash boundary scan + per-chunk SHA-256 +
// known-digest probe, i.e. what happens inside
//
//	writer.WriteEntryReader(entry, tee, size)          internal/pxarmount/commit.go:720, :858
//
// configured by buzhash.NewConfig(4096) (commit.go:302-305) and seeded from the previous
// snapshot's index (commit.go:286-294, :324-329).
//
// NOT COMPILED IN THIS REPOSITORY'S CI: the build image has no Go toolchain (SURVEY.md
// section 0).  The same C symbols are exercised by the Python ctypes tests (tests/) and the
// C++ driver (tests/cxx/).  pxar-mount is built CGO_ENABLED=0 today (.goreleaser.yaml:56);
// this file only builds with `-tags gpu` and CGO_ENABLED=1.
package gpuchunk

/*
#cgo CFLAGS: -I${SRCDIR}/../../include
#cgo LDFLAGS: -L${SRCDIR}/../../pbs_plus_b200 -lpbsgpu -Wl,-rpath,${SRCDIR}/../../pbs_plus_b200
#include <stdlib.h>
#include "pbsgpu.h"
*/
import "C"

import (
	"errors"
	"fmt"
	"io"
	"runtime"
	"unsafe"
)

// Config mirrors buzhash.Config (opaque in the reference; built by NewConfig).
type Config struct{ c C.pbsgpu_cfg }

// NewConfig mirrors buzhash.NewConfig(avgKiB) (commit.go:303 passes 4096 = 4 MiB).
func NewConfig(avgKiB int) (Config, error) {
	var cfg Config
	if rc := C.pbsgpu_config_kib(C.uint32_t(avgKiB), nil, &cfg.c); rc != 0 {
		return cfg, fmt.Errorf("buzhash: invalid average chunk size %d KiB (rc %d)", avgKiB, int(rc))
	}
	return cfg, nil
}

// Engine is one GPU context.  Safe to use from any goroutine: the C side binds the device
// per call and serialises calls per context (no thread-local CUDA state).
type Engine struct{ ctx *C.pbsgpu_ctx }

func Open(device int) (*Engine, error) {
	var ctx *C.pbsgpu_ctx
	if rc := C.pbsgpu_open(C.int(device), &ctx); rc != 0 {
		return nil, fmt.Errorf("pbsgpu_open(%d): rc %d (no CUDA device; there is no CPU fallback)", device, int(rc))
	}
	e := &Engine{ctx}
	runtime.SetFinalizer(e, func(e *Engine) { e.Close() })
	return e, nil
}

func (e *Engine) Close() {
	if e.ctx != nil {
		C.pbsgpu_close(e.ctx)
		e.ctx = nil
	}
}

func (e *Engine) err(rc C.int) error {
	if rc == 0 {
		return nil
	}
	return fmt.Errorf("pbsgpu: %s (rc %d)", C.GoString(C.pbsgpu_strerror(e.ctx)), int(rc))
}

// KnownSet mirrors the session's known-chunk bookkeeping (PreviousBackupRef, commit.go:286-294).
type KnownSet struct {
	e *Engine
	s *C.pbsgpu_set
}

func (e *Engine) NewKnownSet(capacityHint uint64) (*KnownSet, error) {
	var s *C.pbsgpu_set
	if err := e.err(C.pbsgpu_set_create(e.ctx, C.uint64_t(capacityHint), &s)); err != nil {
		return nil, err
	}
	return &KnownSet{e, s}, nil
}

// SeedFromDidx feeds the bytes of the previous .ppxar.didx (origPayloadIdx, commit.go:324-328).
func (k *KnownSet) SeedFromDidx(didx []byte) (uint64, error) {
	if len(didx) == 0 {
		return 0, nil
	}
	var n C.uint64_t
	rc := C.pbsgpu_set_seed_didx(k.s, (*C.uint8_t)(unsafe.Pointer(&didx[0])), C.uint64_t(len(didx)), &n)
	return uint64(n), k.e.err(rc)
}

func (k *KnownSet) Close() { C.pbsgpu_set_destroy(k.s) }

// Chunk is one dynamic-index entry: (end offset, digest) + whether the digest was known.
type Chunk struct {
	Stream uint32
	Known  bool
	End    uint64
	Digest [32]byte
}

// ErrStagingFull is returned by WriteEntryReader when the pinned staging buffer cannot take the entry NOW:
// Flush the batch and write the entry again.
var ErrStagingFull = errors.New("pbsgpu: staging full, call Flush first")

// ErrEntryTooLarge is returned when the entry alone exceeds the staging buffer: flushing cannot help, the entry has
// to go through a Stream / PayloadWriter (which have no size limit).
var ErrEntryTooLarge = errors.New("pbsgpu: entry larger than the staging buffer, use a Stream")

// Batch accumulates whole files in C-owned PINNED staging (Go pointers are never retained by C)
// and pushes them through the GPU in one call -- the batched form of the per-file loop at
// commit.go:604-625 / :697-731.
type Batch struct {
	e    *Engine
	cfg  Config
	buf  unsafe.Pointer
	cap  uint64
	fill uint64
	off  []C.uint64_t
	ln   []C.uint64_t
}

func (e *Engine) NewBatch(cfg Config, stagingBytes uint64) (*Batch, error) {
	p := C.pbsgpu_host_alloc(e.ctx, C.uint64_t(stagingBytes))
	if p == nil {
		return nil, errors.New("pbsgpu: pinned staging allocation failed")
	}
	return &Batch{e: e, cfg: cfg, buf: p, cap: stagingBytes}, nil
}

// WriteEntryReader mirrors transfer.ArchiveWriter.WriteEntryReader(entry, reader, size): it pulls
// exactly size bytes from r (io.ReadFull semantics) into the staging buffer.
func (b *Batch) WriteEntryReader(r io.Reader, size uint64) error {
	if size > b.cap {
		return ErrEntryTooLarge
	}
	start := (b.fill + 255) &^ 255
	if start+size > b.cap {
		return ErrStagingFull
	}
	dst := unsafe.Slice((*byte)(unsafe.Add(b.buf, start)), size)
	if _, err := io.ReadFull(r, dst); err != nil {
		return fmt.Errorf("read payload: %w", err)
	}
	b.off = append(b.off, C.uint64_t(start))
	b.ln = append(b.ln, C.uint64_t(size))
	b.fill = start + size
	return nil
}

// Flush runs scan -> cut -> SHA-256 -> probe for every queued file and returns the chunks in
// (file, offset) order; Known chunks need no upload ("Only new chunks are uploaded").
func (b *Batch) Flush(known *KnownSet) ([]Chunk, error) {
	res, _, err := b.flush(known, false)
	return res, err
}

// FlushWithHashes is Flush plus the XXH3-64 (seed 0) of every queued file, computed on the GPU from the
// same staged bytes: the value emitBackedFile gets from `h := xxh3.New(); io.TeeReader(f, h); h.Sum64()`
// (commit.go:717-725) and stores in ow.backedHashes -- so the host no longer hashes while it reads.
func (b *Batch) FlushWithHashes(known *KnownSet) ([]Chunk, []uint64, error) {
	return b.flush(known, true)
}

func (b *Batch) flush(known *KnownSet, withHashes bool) ([]Chunk, []uint64, error) {
	n := len(b.off)
	if n == 0 {
		return nil, nil, nil
	}
	capChunks := uint64(n)
	for _, l := range b.ln {
		capChunks += uint64(l) / uint64(b.cfg.c.min)
	}
	out := make([]C.pbsgpu_chunk, capChunks+1)
	var nOut C.uint64_t
	var set *C.pbsgpu_set
	if known != nil {
		set = known.s
	}
	var hashes []C.uint64_t
	var hp *C.uint64_t
	if withHashes {
		hashes = make([]C.uint64_t, n)
		hp = &hashes[0]
	}
	rc := C.pbsgpu_chunk_digest_batch_xxh3(b.e.ctx, &b.cfg.c, b.buf, &b.off[0], &b.ln[0], C.uint32_t(n), set,
		&out[0], C.uint64_t(len(out)), &nOut, hp)
	if err := b.e.err(rc); err != nil {
		return nil, nil, err
	}
	res := make([]Chunk, int(nOut))
	for i := range res {
		res[i].Stream = uint32(out[i].stream)
		res[i].Known = out[i].flags&C.PBSGPU_CHUNK_KNOWN != 0
		res[i].End = uint64(out[i].end_off)
		copy(res[i].Digest[:], C.GoBytes(unsafe.Pointer(&out[i].digest[0]), 32))
	}
	var hs []uint64
	if withHashes {
		hs = make([]uint64, n)
		for i := range hashes {
			hs[i] = uint64(hashes[i])
		}
	}
	b.off, b.ln, b.fill = b.off[:0], b.ln[:0], 0
	return res, hs, nil
}

// FileHashes returns the XXH3-64 of every queued file WITHOUT chunking: the verify pass of the commit
// (verifyBackedFileHashes, commit.go:957-976) re-reads the backed files into the staging buffer with
// WriteEntryReader and compares these values with ow.backedHashes.  The queue is cleared.
func (b *Batch) FileHashes() ([]uint64, error) {
	n := len(b.off)
	if n == 0 {
		return nil, nil
	}
	hashes := make([]C.uint64_t, n)
	rc := C.pbsgpu_xxh3_batch(b.e.ctx, b.buf, &b.off[0], &b.ln[0], C.uint32_t(n), &hashes[0])
	if err := b.e.err(rc); err != nil {
		return nil, err
	}
	res := make([]uint64, n)
	for i := range hashes {
		res[i] = uint64(hashes[i])
	}
	b.off, b.ln, b.fill = b.off[:0], b.ln[:0], 0
	return res, nil
}

func (b *Batch) Close() { C.pbsgpu_host_free(b.e.ctx, b.buf) }

// BuildDidx renders the dynamic-index image (<name>.ppxar.didx, commit.go:321-322) for chunks in
// (stream, offset) order; offsets are cumulative over the archive stream, the checksum is computed on the GPU.
func (e *Engine) BuildDidx(chunks []Chunk, uuid [16]byte, ctime int64) ([]byte, error) {
	n := len(chunks)
	rec := make([]C.pbsgpu_chunk, n+1)
	for i, c := range chunks {
		rec[i].stream = C.uint32_t(c.Stream)
		rec[i].end_off = C.uint64_t(c.End)
		for k := 0; k < 32; k++ {
			rec[i].digest[k] = C.uint8_t(c.Digest[k])
		}
	}
	out := make([]byte, uint64(C.pbsgpu_didx_size(C.uint64_t(n))))
	rc := C.pbsgpu_didx_build(e.ctx, &rec[0], C.uint64_t(n), (*C.uint8_t)(unsafe.Pointer(&uuid[0])), C.int64_t(ctime),
		(*C.uint8_t)(unsafe.Pointer(&out[0])), C.uint64_t(len(out)))
	return out, e.err(rc)
}

// BlobCRC32 returns the DataBlob payload checksums of ranges [off[i], off[i]+len[i]) of the batch's pinned
// staging buffer (only NEW chunks need a blob; POST /dynamic_chunk).
func (b *Batch) BlobCRC32(off, length []uint64) ([]uint32, error) {
	n := len(off)
	if n == 0 {
		return nil, nil
	}
	o := make([]C.uint64_t, n)
	l := make([]C.uint64_t, n)
	for i := range off {
		o[i], l[i] = C.uint64_t(off[i]), C.uint64_t(length[i])
	}
	crc := make([]C.uint32_t, n)
	rc := C.pbsgpu_crc32_batch(b.e.ctx, b.buf, &o[0], &l[0], C.uint32_t(n), &crc[0])
	if err := b.e.err(rc); err != nil {
		return nil, err
	}
	res := make([]uint32, n)
	for i := range crc {
		res[i] = uint32(crc[i])
	}
	return res, nil
}

// ---------------------------------------------------------------------------------------------------------------
// Streaming form: ONE byte stream of any length (a VM image, or the whole pxar payload stream), state carried
// across writes -- the literal drop-in for writer.WriteEntryReader(entry, io.Reader, size) (commit.go:718-720).
// ---------------------------------------------------------------------------------------------------------------

// Stream wraps pbsgpu_stream_*.  Bytes travel through a pinned staging ring owned by the C side (reserve -> the
// reader fills it -> commit starts the DMA); Go memory is never retained by C.
type Stream struct {
	e *Engine
	s *C.pbsgpu_stream
}

func (e *Engine) NewStream(cfg Config, known *KnownSet) (*Stream, error) {
	var set *C.pbsgpu_set
	if known != nil {
		set = known.s
	}
	var s *C.pbsgpu_stream
	if err := e.err(C.pbsgpu_stream_open(e.ctx, &cfg.c, set, &s)); err != nil {
		return nil, err
	}
	return &Stream{e, s}, nil
}

// ReadFrom pulls exactly size bytes from r straight into the pinned ring (io.ReadFull per slot), no intermediate copy.
func (st *Stream) ReadFrom(r io.Reader, size uint64) error {
	slot := uint64(C.pbsgpu_stream_slot_bytes(st.s))
	for size > 0 {
		var p unsafe.Pointer
		if err := st.e.err(C.pbsgpu_stream_reserve(st.s, &p)); err != nil {
			return err
		}
		n := size
		if n > slot {
			n = slot
		}
		if _, err := io.ReadFull(r, unsafe.Slice((*byte)(p), n)); err != nil {
			C.pbsgpu_stream_commit(st.s, 0)
			return fmt.Errorf("read payload: %w", err)
		}
		if err := st.e.err(C.pbsgpu_stream_commit(st.s, C.uint64_t(n))); err != nil {
			return err
		}
		size -= n
	}
	return nil
}

// Write implements io.Writer (pageable Go memory is copied into the ring slot by slot).
func (st *Stream) Write(p []byte) (int, error) {
	if len(p) == 0 {
		return 0, nil
	}
	if err := st.e.err(C.pbsgpu_stream_write(st.s, unsafe.Pointer(&p[0]), C.uint64_t(len(p)))); err != nil {
		return 0, err
	}
	return len(p), nil
}

// Suggest registers a suggested boundary at the CURRENT position (call it right before writing a file's PAYLOAD header).
func (st *Stream) Suggest() error {
	return st.e.err(C.pbsgpu_stream_suggest(st.s, C.pbsgpu_stream_position(st.s)))
}

func (st *Stream) Position() uint64 { return uint64(C.pbsgpu_stream_position(st.s)) }

// Poll returns the chunks finished so far (stream order); Finish flushes the final short chunk first.
func (st *Stream) Poll() ([]Chunk, error) {
	var all []Chunk
	buf := make([]C.pbsgpu_chunk, 4096)
	for {
		var n C.uint64_t
		if err := st.e.err(C.pbsgpu_stream_poll(st.s, &buf[0], C.uint64_t(len(buf)), &n)); err != nil {
			return all, err
		}
		if n == 0 {
			return all, nil
		}
		for i := 0; i < int(n); i++ {
			var c Chunk
			c.Known = buf[i].flags&C.PBSGPU_CHUNK_KNOWN != 0
			c.End = uint64(buf[i].end_off)
			copy(c.Digest[:], C.GoBytes(unsafe.Pointer(&buf[i].digest[0]), 32))
			all = append(all, c)
		}
	}
}

func (st *Stream) Finish() ([]Chunk, error) {
	if err := st.e.err(C.pbsgpu_stream_finish(st.s)); err != nil {
		return nil, err
	}
	return st.Poll()
}

func (st *Stream) Close() { C.pbsgpu_stream_close(st.s) }

// PayloadWriter produces the pxar v2 PAYLOAD stream the production chunker sees -- start marker, then per file a
// 16-byte PAYLOAD header + content (internal/pxarmount/pxarfs.go:408-411) -- through ONE Stream, with a suggested
// boundary at every file start.  WriteEntryReader returns the entry's payload offset (what the mpxar PAYLOAD_REF
// stores).  This, not per-file batching, is the layout an existing .ppxar.didx describes.
type PayloadWriter struct {
	st      *Stream
	Chunks  []Chunk
	started bool
}

const (
	pxarPayload            = 0x28147a1b0b7c1a25
	pxarPayloadStartMarker = 0x834c68c2194a4ed2
	pxarPayloadTailMarker  = 0x6c72b78b984c81b5
)

func header(htype, fullSize uint64) []byte {
	var h [16]byte
	for i := 0; i < 8; i++ {
		h[i] = byte(htype >> (8 * i))
		h[8+i] = byte(fullSize >> (8 * i))
	}
	return h[:]
}

func (e *Engine) NewPayloadWriter(cfg Config, known *KnownSet) (*PayloadWriter, error) {
	st, err := e.NewStream(cfg, known)
	if err != nil {
		return nil, err
	}
	w := &PayloadWriter{st: st}
	_, err = st.Write(header(pxarPayloadStartMarker, 16))
	return w, err
}

func (w *PayloadWriter) WriteEntryReader(r io.Reader, size uint64) (payloadOffset uint64, err error) {
	payloadOffset = w.st.Position()
	if err = w.st.Suggest(); err != nil {
		return
	}
	if _, err = w.st.Write(header(pxarPayload, 16+size)); err != nil {
		return
	}
	if err = w.st.ReadFrom(r, size); err != nil {
		return
	}
	done, err := w.st.Poll()
	w.Chunks = append(w.Chunks, done...)
	return
}

func (w *PayloadWriter) Finish() ([]Chunk, error) {
	if _, err := w.st.Write(header(pxarPayloadTailMarker, 16)); err != nil {
		return nil, err
	}
	done, err := w.st.Finish()
	w.Chunks = append(w.Chunks, done...)
	w.st.Close()
	return w.Chunks, err
}

// ---------------------------------------------------------------------------------------------------------------
// Multi-GPU: one Engine per GPU (one goroutine each), files sharded by range; the ONE exchange step.
// ---------------------------------------------------------------------------------------------------------------

// NcclComm is an ncclComm_t made through the C ABI's helpers; a caller with its own NCCL binding passes its
// communicator to AllGather through NcclCommFromHandle instead.
type NcclComm struct{ h unsafe.Pointer }

func NcclUniqueID() ([128]byte, error) {
	var id [128]byte
	if rc := C.pbsgpu_nccl_unique_id((*C.uint8_t)(unsafe.Pointer(&id[0]))); rc != 0 {
		return id, fmt.Errorf("pbsgpu: NCCL unavailable (rc %d)", int(rc))
	}
	return id, nil
}

func (e *Engine) NewNcclComm(id [128]byte, nranks, rank int) (*NcclComm, error) {
	var h unsafe.Pointer
	if err := e.err(C.pbsgpu_nccl_comm_create(e.ctx, (*C.uint8_t)(unsafe.Pointer(&id[0])), C.int(nranks), C.int(rank), &h)); err != nil {
		return nil, err
	}
	return &NcclComm{h}, nil
}

func NcclCommFromHandle(h unsafe.Pointer) *NcclComm { return &NcclComm{h} }
func (c *NcclComm) Close()                           { C.pbsgpu_nccl_comm_destroy(c.h) }

// AllGather merges this rank's chunk digests with every other rank's (pbsgpu_set_allgather: counts + padded
// digests over NCCL/NVLink, then every replica inserts all of them in global (rank, index) order) and sets
// Known on the chunks that are known globally.  Collective: every rank calls it once per batch.
func (k *KnownSet) AllGather(comm *NcclComm, chunks []Chunk) error {
	n := len(chunks)
	dig := make([]byte, 32*n+1)
	hit := make([]byte, n+1)
	for i := range chunks {
		copy(dig[32*i:], chunks[i].Digest[:])
	}
	rc := C.pbsgpu_set_allgather(k.s, comm.h, (*C.uint8_t)(unsafe.Pointer(&dig[0])), C.uint64_t(n), (*C.uint8_t)(unsafe.Pointer(&hit[0])))
	if err := k.e.err(rc); err != nil {
		return err
	}
	for i := range chunks {
		chunks[i].Known = hit[i] != 0
	}
	return nil
}

// BlobEncode renders complete uncompressed DataBlobs (magic | crc32 | payload) for ranges of the batch's staging
// buffer -- the upload bodies of the NEW chunks (POST /dynamic_chunk, internal/server/backup/log_cleanup.go:19-31).
func (b *Batch) BlobEncode(off, length []uint64) ([][]byte, error) {
	n := len(off)
	if n == 0 {
		return nil, nil
	}
	o := make([]C.uint64_t, n)
	l := make([]C.uint64_t, n)
	oo := make([]C.uint64_t, n)
	var total uint64
	for i := range off {
		o[i], l[i], oo[i] = C.uint64_t(off[i]), C.uint64_t(length[i]), C.uint64_t(total)
		total += uint64(C.pbsgpu_blob_size(C.uint64_t(length[i])))
	}
	out := make([]byte, total+1)
	rc := C.pbsgpu_blob_encode_batch(b.e.ctx, b.buf, &o[0], &l[0], C.uint32_t(n), (*C.uint8_t)(unsafe.Pointer(&out[0])), &oo[0], nil)
	if err := b.e.err(rc); err != nil {
		return nil, err
	}
	res := make([][]byte, n)
	for i := range off {
		res[i] = out[uint64(oo[i]) : uint64(oo[i])+12+length[i]]
	}
	return res, nil
}

// BlobEncodeZ is BlobEncode with the zstd-compressed DataBlob form where that is smaller (upstream DataBlob::encode
// keeps a compressed payload only then).  The frames are built on the GPU from RLE and raw blocks -- they remove
// the zero runs of disk images and sparse files; data without such runs stays uncompressed.
func (b *Batch) BlobEncodeZ(off, length []uint64) ([][]byte, error) {
	return b.blobEncodeZstd(off, length, false)
}

// BlobEncodeLZ is BlobEncodeZ whose frames also hold zstd Compressed_Blocks from the GPU's greedy LZ parse wherever
// those are smaller than the block: text, logs and repeated records shrink too.  It costs more GPU time per byte than
// BlobEncodeZ and compresses less than zstd level 1 (no Huffman literals, predefined FSE tables, block-local matches).
func (b *Batch) BlobEncodeLZ(off, length []uint64) ([][]byte, error) {
	return b.blobEncodeZstd(off, length, true)
}

func (b *Batch) blobEncodeZstd(off, length []uint64, lz bool) ([][]byte, error) {
	n := len(off)
	if n == 0 {
		return nil, nil
	}
	o := make([]C.uint64_t, n)
	l := make([]C.uint64_t, n)
	oo := make([]C.uint64_t, n)
	ol := make([]C.uint64_t, n)
	var total uint64
	for i := range off {
		o[i], l[i], oo[i] = C.uint64_t(off[i]), C.uint64_t(length[i]), C.uint64_t(total)
		total += uint64(C.pbsgpu_blob_size(C.uint64_t(length[i])))
	}
	out := make([]byte, total+1)
	var rc C.int
	if lz {
		rc = C.pbsgpu_blob_encode_batch_lz(b.e.ctx, b.buf, &o[0], &l[0], C.uint32_t(n), (*C.uint8_t)(unsafe.Pointer(&out[0])), &oo[0], &ol[0], nil)
	} else {
		rc = C.pbsgpu_blob_encode_batch_z(b.e.ctx, b.buf, &o[0], &l[0], C.uint32_t(n), (*C.uint8_t)(unsafe.Pointer(&out[0])), &oo[0], &ol[0], nil)
	}
	if err := b.e.err(rc); err != nil {
		return nil, err
	}
	res := make([][]byte, n)
	for i := range off {
		res[i] = out[uint64(oo[i]) : uint64(oo[i])+uint64(ol[i])]
	}
	return res, nil
}
