"""pbsgpu_blob_encode_batch_lz (K9, csrc/zlz.cu) on the GPU: bit-exact against the restated encoder
(oracle/zstd_lz.py blob_encode_lz), CRCs against zlib, every compressed payload read back by libzstd (pyarrow)."""
import zlib

import numpy as np
import pytest

import pbs_plus_b200 as pg
from oracle import pyref, zstd_lz
from pbs_plus_b200 import transfer

pytestmark = pytest.mark.gpu
B = pyref.ZFRAME_BLOCK


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


@pytest.fixture(scope="module")
def eng():
    e = pg.Engine(0)
    yield e
    e.close()


def rnd(n, seed):
    return np.random.default_rng(seed).integers(0, 256, size=n, dtype=np.uint8)


def text(nbytes, seed):
    return np.frombuffer(zstd_lz.text_corpus(seed, nbytes), dtype=np.uint8)


def to_dev(torch, a):
    return torch.from_numpy(np.array(a)).to("cuda")


def decode(frame, size):
    pa = pytest.importorskip("pyarrow")
    return pa.Codec("zstd").decompress(frame, decompressed_size=size).to_pybytes() if size else b""


def pack(parts, lead=3):
    """Concatenated parts behind `lead` filler bytes: every source misaligned."""
    ln = np.array([len(p) for p in parts], dtype=np.uint64)
    off = np.zeros(len(parts), dtype=np.uint64)
    np.cumsum(ln[:-1], out=off[1:])
    buf = np.concatenate([np.full(lead, 0xEE, np.uint8)] + list(parts) + [np.zeros(1, np.uint8)])
    return buf, off + np.uint64(lead), ln


def matrix():
    periodic = [np.resize(rnd(p, p), 400_000) for p in (1, 2, 3, 7, 1000, 1025, 4096)]
    return [np.zeros(0, np.uint8), rnd(1, 1), rnd(2, 2), rnd(3, 3), rnd(4, 4),
            rnd(300_000, 5),                                                   # random: raw
            np.concatenate([np.zeros(3 * B, np.uint8), np.full(B + 5, 7, np.uint8)]),   # RLE blocks
            *periodic,
            np.resize(rnd(1000, 6), 1000 + B)[:B],                             # a match that ends at the block end
            np.concatenate([rnd(1000, 7), np.zeros(3 * B - 10, np.uint8), rnd(B - 777, 8)]),   # zero run off the grid
            np.resize(rnd(5000, 9), 2 * B + 13),                               # ragged tail
            text(1 << 20, 10)]


def check_blobs(parts, blobs, crc, want=None):
    for i, (blob, p) in enumerate(zip(blobs, parts)):
        if want is not None:
            assert blob == want[i], (i, len(blob), len(want[i]))
        assert int.from_bytes(blob[8:12], "little") == zlib.crc32(blob[12:]) == int(crc[i])
        if blob[:8] == pyref.BLOB_MAGIC_COMPRESSED:
            assert len(blob) < 12 + len(p) and decode(blob[12:], len(p)) == p.tobytes()
        else:
            assert blob[:8] == pyref.BLOB_MAGIC_UNCOMPRESSED and blob[12:] == p.tobytes()


def test_blob_encode_batch_lz_matches_the_oracle(eng, torch):
    parts = matrix()
    want = [zstd_lz.blob_encode_lz(p.tobytes()) for p in parts]
    buf, off, ln = pack(parts)
    for base in (buf, to_dev(torch, buf)):
        blobs, crc = eng.blob_encode_batch_lz(base, off, ln)
        check_blobs(parts, blobs, crc, want)
    z, _ = eng.blob_encode_batch_z(buf, off, ln)
    assert all(len(a) <= len(b) for a, b in zip(blobs, z))
    assert blobs[5] == z[5]                                                    # random data: the same blob as _z


def test_blob_encode_batch_lz_on_chunker_output(eng, torch):
    """The NEW chunks of a mixed image (text, random data, zero runs) chunked on the GPU and encoded in one call."""
    img = rnd(24 << 20, 20)
    img[2 << 20: 8 << 20] = text(6 << 20, 21)
    img[(11 << 20) + 4321: (15 << 20) + 99] = 0
    img[17 << 20: 19 << 20] = np.resize(text(1 << 16, 22), 2 << 20)
    d = to_dev(torch, img)
    rec = eng.chunk_digest_batch(pg.make_config(1 << 20), d, [0], [len(img)])
    ends = rec["end_off"].astype(np.uint64)
    starts = np.concatenate([[0], ends[:-1]]).astype(np.uint64)
    blobs, crc = eng.blob_encode_batch_lz(d, starts, ends - starts)
    z, _ = eng.blob_encode_batch_z(d, starts, ends - starts)
    parts = [img[int(s0): int(e0)] for s0, e0 in zip(starts, ends)]
    check_blobs(parts, blobs, crc, [zstd_lz.blob_encode_lz(p.tobytes()) for p in parts])
    assert all(len(a) <= len(b) for a, b in zip(blobs, z))
    assert sum(map(len, blobs)) < sum(map(len, z))


def test_dedup_writer_lz_uploads_oracle_blobs(eng):
    blobs = []
    w = transfer.NewRemoteDedupSplitArchiveWriter(eng, pg.make_config(1 << 16), known=eng.digest_set(),
                                                  upload_blob=lambda d, b: blobs.append((d, b)), blob_codec="lz")
    log = text(3_000_000, 30)
    mixed = rnd(2_000_000, 31)
    mixed[500_000:1_500_000] = 0
    files = [("app.log", log), ("copy.log", log.copy()), ("disk.img", mixed), ("small", rnd(100, 32))]
    for name, data in files:
        w.WriteEntry(transfer.Entry(name, len(data)), data.tobytes())
    w.Finish()
    import oracle
    ref = oracle.chunk_digest_streams(oracle.config(1 << 16), [d for _, d in files])
    want, seen, start = [], set(), {}
    for r in ref:
        i = int(r["stream"]); s0 = start.get(i, 0); e0 = int(r["end_off"]); start[i] = e0
        dg = bytes(r["digest"])
        if dg not in seen:
            seen.add(dg)
            want.append((dg, zstd_lz.blob_encode_lz(files[i][1][s0:e0].tobytes())))
    assert blobs == want
    assert sum(b[:8] == pyref.BLOB_MAGIC_COMPRESSED for _, b in blobs) > len(blobs) // 2


def test_blob_codec_is_checked(eng):
    with pytest.raises(ValueError):
        transfer.DedupWriter(eng, pg.make_config(1 << 16), blob_codec="zstd")


def test_blob_encode_batch_lz_over_1_gib_resident(eng, torch):
    """1.25 GiB of device-resident compressible data (text tiles, zero runs, random stretches) in 4 MiB chunks: every CRC
    equals zlib's, and libzstd decodes a spread sample of the frames -- several of K9's passes, so its per-pass scratch
    is reused."""
    n, CH = 5 << 28, 4 << 20
    tile = to_dev(torch, text(16 << 20, 40))
    d = tile.repeat(n // tile.numel())
    d[(1 << 30) + 12345: (1 << 30) + (64 << 20)] = 0
    d[200 << 20: 232 << 20] = to_dev(torch, rnd(32 << 20, 41))
    off = np.arange(0, n, CH, dtype=np.uint64)
    ln = np.full(len(off), CH, dtype=np.uint64)
    ln[-1] -= np.uint64(777)                                                   # a ragged last chunk
    blobs, crc = eng.blob_encode_batch_lz(d, off, ln)
    for i, blob in enumerate(blobs):
        assert int.from_bytes(blob[8:12], "little") == zlib.crc32(blob[12:]) == int(crc[i])
    host = d.cpu().numpy()
    for i in list(range(0, len(off), 17)) + [len(off) - 1, 50, 51, 256]:
        p = host[int(off[i]): int(off[i] + ln[i])]
        blob = blobs[i]
        if blob[:8] == pyref.BLOB_MAGIC_COMPRESSED:
            assert decode(blob[12:], len(p)) == p.tobytes(), i
        else:
            assert blob[12:] == p.tobytes(), i
    assert sum(map(len, blobs)) < n * 0.8
