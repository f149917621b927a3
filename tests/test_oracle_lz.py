"""The restated zstd match stage (oracle/zstd_lz.py: zstd_compressed_block, lz_parse, zstd_frame_lz, blob_encode_lz)
against an independent decoder: pyarrow's zstd codec links libzstd, which must read every frame back to its input."""
import zlib

import numpy as np
import pytest

from oracle import pyref, zstd_lz

pa = pytest.importorskip("pyarrow")
B = pyref.ZFRAME_BLOCK


def decode(frame: bytes, size: int) -> bytes:
    return pa.Codec("zstd").decompress(frame, decompressed_size=size).to_pybytes() if size else b""


def rnd(n, seed):
    return np.random.default_rng(seed).integers(0, 256, size=n, dtype=np.uint8).tobytes()


def one_block_frame(spec, trailing, seed):
    """A frame of one Compressed_Block from (literal length, offset, match length) triples; offsets are clamped to the
    output so far.  Returns (frame, expected output)."""
    rng = np.random.default_rng(seed)
    lits = rng.integers(0, 256, size=sum(s[0] for s in spec) + trailing, dtype=np.uint8).tobytes()
    out, li, seqs = bytearray(), 0, []
    for ll, of, ml in spec:
        out += lits[li:li + ll]
        li += ll
        of = min(of, len(out))
        for _ in range(ml):
            out.append(out[-of])
        seqs.append((ll, of, ml))
    out += lits[li:]
    body = zstd_lz.zstd_compressed_block(lits, seqs)
    # a Compressed_Block must be smaller than min(window, 128 KiB); the Single_Segment window is the content
    assert len(out) <= B and len(body) < len(out)
    frame = b"\x28\xb5\x2f\xfd\xe0" + len(out).to_bytes(8, "little") + (1 | (2 << 1) | (len(body) << 3)).to_bytes(3, "little")
    return frame + body, bytes(out)


def check_blocks(specs, trailing=3, seed=0):
    for k, spec in enumerate(specs):
        frame, want = one_block_frame(spec, trailing, seed + k)
        assert decode(frame, len(want)) == want, (k, spec[:4])


def code_values(codes, cap):
    """Both ends of every code's range, capped."""
    return sorted({min(v, cap) for base, bits in codes for v in (base, base + (1 << bits) - 1)})


def test_every_literal_length_code():
    # the first sequence builds no history (literal length >= 1); the match behind each literal run makes the block
    # larger than its content
    specs = [[(ll, 1, max(3, ll // 2 + 16))] for ll in code_values(zstd_lz.LL_CODES, 80_000) if ll]
    specs.append([(1, 1, 5), (0, 1, 3), (0, 1, 4)])                    # literal length 0
    check_blocks(specs)


def test_every_match_length_code():
    specs = [[(1, 1, ml), (2, 1, 3), (0, 1, 64)] for ml in code_values(zstd_lz.ML_CODES, 120_000)]
    check_blocks(specs)


def test_offsets_up_to_128_kib():
    specs = []
    for of in [1, 2, 3, 4, 5, 7, 8, 100, 1000, 4095, 4096, 65535, 65536, 100_000, 126_000, 130_000]:
        hist = max(of, 8)
        specs.append([(5, 1, hist), (7, of, 6), (0, of, 300)])          # history by a run, then matches at offset `of`
    check_blocks(specs, trailing=0)


def test_literal_header_and_sequence_count_forms():
    specs = []
    for n_lit in (31, 32, 4095, 4096, 40_000):                          # 1-, 2- and 3-byte Raw_Literals headers
        specs.append([(n_lit, 1, n_lit + 64)])
    for nseq in (1, 127, 128, 0x7EFF, 0x7F00, 0x7F00 + 300):             # 1-, 2- and 3-byte Number_of_Sequences
        specs.append([(1, 1, 300)] + [(0, 1, 3)] * (nseq - 1))
    check_blocks(specs)


def lz_cases():
    periodic = {f"period {p}": (rnd(p, p) * (400_000 // p + 1))[:400_000] for p in (1, 2, 3, 7, 1000, 1025, 4096)}
    return {
        "empty": b"", "1 byte": b"a", "2 bytes": b"ab", "3 bytes": b"abc", "4 bytes": b"abcd",
        "random": rnd(300_000, 1),
        "constant blocks": bytes(3 * B) + b"\x07" * (B + 5),
        **periodic,
        # a block that ends inside a match: the match is capped at the block end
        "match to block end": rnd(1000, 2) + rnd(1000, 2) * (B // 1000 + 1),
        "zero run off the grid": rnd(1000, 3) + bytes(3 * B - 10) + rnd(B - 777, 4),
        "ragged tail": (rnd(5000, 5) * 100)[:2 * B + 13],
        "text": zstd_lz.text_corpus(7, 1 << 20),
    }


@pytest.mark.parametrize("name", list(lz_cases()))
def test_frame_lz_is_read_by_libzstd(name):
    data = lz_cases()[name]
    frame = zstd_lz.zstd_frame_lz(data)
    assert decode(frame, len(data)) == data
    blob, blob_z = zstd_lz.blob_encode_lz(data), pyref.blob_encode(data)
    assert len(blob) <= len(blob_z)
    assert int.from_bytes(blob[8:12], "little") == zlib.crc32(blob[12:])
    if name == "random":
        assert blob == blob_z and frame == pyref.zstd_frame_rle_raw(data)
    if name.startswith("period") and name != "period 1":
        assert len(frame) < len(pyref.zstd_frame_rle_raw(data)) // 20
    if name == "text":
        assert len(frame) < len(data) * 0.8


def test_frame_lz_blocks_are_local():
    """A block equal to the one before it gains nothing: matches never reach into an earlier block."""
    blk = rnd(B, 9)
    assert zstd_lz.zstd_frame_lz(blk * 2) == pyref.zstd_frame_rle_raw(blk * 2)


def test_text_ratio_next_to_libzstd_level_1(capsys):
    data = zstd_lz.text_corpus(11, 1 << 20)
    ours = len(data) / len(zstd_lz.zstd_frame_lz(data))
    lvl1 = len(data) / len(pa.Codec("zstd", compression_level=1).compress(data))
    with capsys.disabled():
        print(f"\ntext corpus 1 MiB: greedy LZ frame ratio {ours:.2f}, libzstd level 1 {lvl1:.2f}")
    assert ours > 1.0
