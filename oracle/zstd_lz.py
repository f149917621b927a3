"""oracle/zstd_lz.py -- restatement of the DataBlob zstd match stage (K9, csrc/zlz.cu) in numpy / pure Python.

TEST INFRASTRUCTURE.  The GPU must agree with it bit for bit; libzstd (pyarrow) decodes its frames in the tests.
The frame, block grid, RLE rule and DataBlob layout are those of oracle/pyref.py (zstd_frame_rle_raw, blob_encode),
which this module builds on.
"""
from __future__ import annotations

import bisect
import zlib

import numpy as np

from .pyref import BLOB_MAGIC_COMPRESSED, BLOB_MAGIC_UNCOMPRESSED, ZFRAME_BLOCK

# -- f3, match stage (K9, csrc/zlz.cu): a zstd frame whose non-constant blocks are Compressed_Blocks built from a greedy,
#    block-local LZ parse, Raw_Literals and Predefined_Mode FSE sequences (RFC 8878 3.1.1.3).  The GPU must agree with
#    this bit for bit; libzstd decodes both in the tests. ----------------------------------------------------------------
LZ_HLOG, LZ_SEG, LZ_MINMATCH = 14, 1024, 4

# Predefined distributions (RFC 8878 3.1.1.3.2.2); -1 = "less than 1"
LL_NORM = [4, 3, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 1, 1, 1, 2, 2, 2, 2, 2, 2, 2, 2, 2, 3, 2, 1, 1, 1, 1, 1, -1, -1, -1, -1]
ML_NORM = [1, 4, 3, 2, 2, 2, 2, 2, 2] + [1] * 37 + [-1] * 7
OF_NORM = [1, 1, 1, 1, 1, 1, 2, 2, 2] + [1] * 15 + [-1] * 5
LL_LOG, ML_LOG, OF_LOG = 6, 6, 5
# code -> (baseline, extra bits)
LL_CODES = [(i, 0) for i in range(16)] + list(zip(
    [16, 18, 20, 22, 24, 28, 32, 40, 48, 64, 128, 256, 512, 1024, 2048, 4096, 8192, 16384, 32768, 65536],
    [1, 1, 1, 1, 2, 2, 3, 3, 4, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16]))
ML_CODES = [(i + 3, 0) for i in range(32)] + list(zip(
    [35, 37, 39, 41, 43, 47, 51, 59, 67, 83, 99, 131, 259, 515, 1027, 2051, 4099, 8195, 16387, 32771, 65539],
    [1, 1, 1, 1, 2, 2, 3, 3, 4, 4, 5, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16]))


def fse_decode_table(norm, log):
    """RFC 8878 4.1.1: per state (symbol, nbBits, baseline)."""
    size = 1 << log
    sym = [0] * size
    high = size - 1
    for s, p in enumerate(norm):
        if p == -1:
            sym[high] = s
            high -= 1
    pos, step = 0, (size >> 1) + (size >> 3) + 3
    for s, p in enumerate(norm):
        for _ in range(max(p, 0)):
            sym[pos] = s
            pos = (pos + step) & (size - 1)
            while pos > high:
                pos = (pos + step) & (size - 1)
    nxt = [1 if p == -1 else p for p in norm]
    table = []
    for u in range(size):
        s = sym[u]
        x = nxt[s]
        nxt[s] += 1
        nb = log - (x.bit_length() - 1)
        table.append((s, nb, (x << nb) - size))
    return table


def fse_encode_table(norm, log):
    """enc[s][S'] = the state X of symbol s whose [baseline, baseline + 2^nbBits) holds S' (the decoder's next state)."""
    size = 1 << log
    enc = [[-1] * size for _ in norm]
    for x, (s, nb, base) in enumerate(fse_decode_table(norm, log)):
        for t in range(base, base + (1 << nb)):
            enc[s][t] = x
    return enc


_FSE = None


def _fse():
    global _FSE
    if _FSE is None:
        _FSE = [(fse_decode_table(n, lg), fse_encode_table(n, lg), lg)
                for n, lg in ((LL_NORM, LL_LOG), (ML_NORM, ML_LOG), (OF_NORM, OF_LOG))]
    return _FSE


def zstd_compressed_block(literals: bytes, sequences) -> bytes:
    """Block_Content of a Compressed_Block (no Block_Header): Raw_Literals_Block of `literals`, then the sequences
    (literal length, offset, match length) with all three symbol types in Predefined_Mode and no repeat offsets."""
    literals = bytes(literals)
    n_lit, n = len(literals), len(sequences)
    if n_lit <= 31:
        out = bytearray([n_lit << 3])
    elif n_lit <= 4095:
        out = bytearray((0b0100 | (n_lit << 4)).to_bytes(2, "little"))
    else:
        out = bytearray((0b1100 | (n_lit << 4)).to_bytes(3, "little"))
    out += literals
    if n < 128:
        out.append(n)
    elif n < 0x7F00:
        out += bytes([(n >> 8) + 128, n & 0xFF])
    else:
        out += bytes([255]) + (n - 0x7F00).to_bytes(2, "little")
    if n == 0:
        return bytes(out)
    out.append(0)   # Symbol_Compression_Modes: LL, OF, ML predefined
    (ll_dec, ll_enc, ll_log), (ml_dec, ml_enc, ml_log), (of_dec, of_enc, of_log) = _fse()
    ll = np.array([q[0] for q in sequences], dtype=np.int64)
    of = np.array([q[1] for q in sequences], dtype=np.int64)
    ml = np.array([q[2] for q in sequences], dtype=np.int64)
    assert ll.min() >= 0 and of.min() >= 1 and ml.min() >= 3
    llb, mlb = np.array(LL_CODES), np.array(ML_CODES)
    llc = np.searchsorted(llb[:, 0], ll, side="right") - 1
    mlc = np.searchsorted(mlb[:, 0], ml, side="right") - 1
    ofv = of + 3
    ofc = np.floor(np.log2(ofv)).astype(np.int64)
    ofc -= (1 << ofc) > ofv                                  # guard the float rounding of log2
    ofc += (2 << ofc) <= ofv
    syms = list(zip(llc.tolist(), (ll - llb[llc, 0]).tolist(), llb[llc, 1].tolist(), mlc.tolist(),
                    (ml - mlb[mlc, 0]).tolist(), mlb[mlc, 1].tolist(), ofc.tolist(), (ofv - (1 << ofc)).tolist()))
    bits = bytearray()
    acc, nbits = 0, 0

    def put(v, nb):   # forward bitstream, LSB first
        nonlocal acc, nbits
        acc |= (v & ((1 << nb) - 1)) << nbits
        nbits += nb
        if nbits >= 64:
            bits.extend((acc & ((1 << 64) - 1)).to_bytes(8, "little"))
            acc >>= 64
            nbits -= 64

    llc, llx, llb, mlc, mlx, mlb, ofc, ofx = syms[-1]
    # the last sequence starts from the lowest state of each of its symbols
    s_ll = next(x for x, e in enumerate(ll_dec) if e[0] == llc)
    s_ml = next(x for x, e in enumerate(ml_dec) if e[0] == mlc)
    s_of = next(x for x, e in enumerate(of_dec) if e[0] == ofc)
    put(llx, llb); put(mlx, mlb); put(ofx, ofc)
    for k in range(n - 2, -1, -1):
        llc, llx, llb, mlc, mlx, mlb, ofc, ofx = syms[k]
        x = of_enc[ofc][s_of]; put(s_of - of_dec[x][2], of_dec[x][1]); s_of = x
        x = ml_enc[mlc][s_ml]; put(s_ml - ml_dec[x][2], ml_dec[x][1]); s_ml = x
        x = ll_enc[llc][s_ll]; put(s_ll - ll_dec[x][2], ll_dec[x][1]); s_ll = x
        put(llx, llb); put(mlx, mlb); put(ofx, ofc)
    put(s_ml, ml_log); put(s_of, of_log); put(s_ll, ll_log)
    put(1, 1)
    out += bits + acc.to_bytes((nbits + 7) // 8, "little")
    return bytes(out)


def lz_parse(block: bytes):
    """The greedy parse of one block -> (literals, [(literal length, offset, match length)]), trailing literals
    included in `literals`.  cand(p) = the last earlier-segment position with the same 14-bit hash; a match starts
    where the 4 bytes there agree and runs as far as the bytes agree."""
    S = len(block)
    if S < LZ_MINMATCH:
        return block, []
    a = np.frombuffer(block, dtype=np.uint8)
    u = (a[:-3].astype(np.uint32) | (a[1:-2].astype(np.uint32) << 8) | (a[2:-1].astype(np.uint32) << 16)
         | (a[3:].astype(np.uint32) << 24))                     # u32le at every p <= S - 4
    h = ((u * np.uint32(0x9E3779B1)) >> np.uint32(32 - LZ_HLOG)).astype(np.int64)
    pos = np.arange(len(u), dtype=np.int64)
    keys = h * S + pos                                          # sorted: by hash, then position
    order = np.argsort(keys, kind="stable")
    ks = keys[order]
    i = np.searchsorted(ks, h * S + (pos // LZ_SEG) * LZ_SEG, side="left") - 1
    ok = i >= 0
    cand = np.where(ok, ks[np.maximum(i, 0)] - h * S, -1)
    ok &= (cand >= 0) & (cand < (pos // LZ_SEG) * LZ_SEG)
    cand = np.where(ok, cand, -1)
    m = ok & (u[np.maximum(cand, 0)] == u)
    starts = np.nonzero(m)[0].tolist()
    cand = cand.tolist()
    lits, seqs = bytearray(), []
    p, j = 0, 0
    while True:
        j = bisect.bisect_left(starts, p, j)
        if j >= len(starts):
            break
        q = starts[j]
        c = cand[q]
        L, w = 4, 16
        while q + L < S:   # longest common prefix: the window doubles while it matches and halves on a mismatch
            w = min(w, S - q - L)
            if block[c + L:c + L + w] == block[q + L:q + L + w]:
                L += w
                w *= 2
            elif w == 1:
                break
            else:
                w //= 2
        lits += block[p:q]
        seqs.append((q - p, q - c, L))
        p = q + L
    lits += block[p:]
    return bytes(lits), seqs


def zstd_frame_lz(data: bytes) -> bytes:
    """zstd_frame_rle_raw's frame and block grid, with every non-constant block the Compressed_Block of its greedy parse
    where that is smaller than the block (ties and blocks without a match stay Raw_Blocks)."""
    data = bytes(data)
    out = bytearray(b"\x28\xb5\x2f\xfd\xe0" + len(data).to_bytes(8, "little"))
    nb = max(1, (len(data) + ZFRAME_BLOCK - 1) // ZFRAME_BLOCK)
    for b in range(nb):
        blk = data[b * ZFRAME_BLOCK:(b + 1) * ZFRAME_BLOCK]
        last = int(b + 1 == nb)
        if len(blk) > 0 and blk.count(blk[:1]) == len(blk):
            out += (last | (1 << 1) | (len(blk) << 3)).to_bytes(3, "little") + blk[:1]
            continue
        lits, seqs = lz_parse(blk)
        body = zstd_compressed_block(lits, seqs) if seqs else None
        if body is not None and len(body) < len(blk):
            out += (last | (2 << 1) | (len(body) << 3)).to_bytes(3, "little") + body
        else:
            out += (last | (len(blk) << 3)).to_bytes(3, "little") + blk
    return bytes(out)


def blob_encode_lz(data: bytes) -> bytes:
    """blob_encode with zstd_frame_lz's frame: the compressed blob when the frame is smaller than the data."""
    data = bytes(data)
    if data:
        fr = zstd_frame_lz(data)
        if len(fr) < len(data):
            return BLOB_MAGIC_COMPRESSED + zlib.crc32(fr).to_bytes(4, "little") + fr
    return BLOB_MAGIC_UNCOMPRESSED + zlib.crc32(data).to_bytes(4, "little") + data


def text_corpus(seed: int, nbytes: int) -> bytes:
    """Seeded text-like bytes: words of 2..9 lowercase letters from a 4096-word splitmix64 vocabulary, drawn with a
    skewed (roughly Zipf-like) frequency, separated by spaces, with a newline every 16th word."""
    def mix(x):
        with np.errstate(over="ignore"):
            x = x + np.uint64(0x9E3779B97F4A7C15)
            z = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
            z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))

    V = 4096
    r = mix(np.arange(V * 10, dtype=np.uint64) + np.uint64(seed * 0x1000003))
    vocab = []
    for w in range(V):
        k = 2 + int(r[w * 10] % np.uint64(8))
        vocab.append(bytes((97 + (r[w * 10 + 1: w * 10 + 1 + k] % np.uint64(26))).astype(np.uint8)))
    n_words = nbytes // 4 + 16
    u = (mix(np.arange(n_words, dtype=np.uint64) + np.uint64(seed) * np.uint64(0x10000000000)) >> np.uint64(11)).astype(
        np.float64) / float(1 << 53)
    idx = np.minimum((V * u ** 3).astype(np.int64), V - 1)
    seps = [b"\n" if i % 16 == 15 else b" " for i in range(16)]
    out = b"".join(vocab[i] + seps[j & 15] for j, i in enumerate(idx.tolist()))
    while len(out) < nbytes:
        out += out
    return out[:nbytes]
