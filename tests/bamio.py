"""Minimal BGZF/BAM writer for the tests (SAM/BAM spec v1 section 4). Sequence and qualities are
omitted (l_seq = 0); the hot path never looks at them."""
from __future__ import annotations

import struct
import zlib

import numpy as np

_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def _bgzf_block(data: bytes, level: int = 1) -> bytes:
    co = zlib.compressobj(level, zlib.DEFLATED, -15)
    comp = co.compress(data) + co.flush()
    bsize = len(comp) + 26
    assert bsize <= 65536
    hdr = struct.pack("<BBBBIBBHBBHH", 31, 139, 8, 4, 0, 0, 255, 6, ord("B"), ord("C"), 2, bsize - 1)
    return hdr + comp + struct.pack("<II", zlib.crc32(data) & 0xFFFFFFFF, len(data))


def reg2bin(beg: int, end: int) -> int:
    end -= 1
    for shift, base in ((14, 4681), (17, 585), (20, 73), (23, 9), (26, 1)):
        if beg >> shift == end >> shift:
            return base + (beg >> shift)
    return 0


def encode_record(tid, pos, mapq, flag, cigar_words, name=b"r", hp=None, hp_type="C", sa=None, end=None, extra_aux=b""):
    cig = np.asarray(cigar_words, dtype=np.uint32)
    aux = b""
    l_seq = 0
    if len(cig) > 65535:
        # long CIGAR convention: <l_seq>S<rlen>N in the record, real CIGAR in CG:B,I
        ops = cig & 15
        rlen = int((cig >> 4)[np.isin(ops, [0, 2, 3, 7, 8])].sum())
        aux += b"CGBI" + struct.pack("<I", len(cig)) + cig.astype("<u4").tobytes()
        cig = np.asarray([(l_seq << 4) | 4, (rlen << 4) | 3], dtype=np.uint32)
    if hp is not None:
        fmt = {"C": "<B", "c": "<b", "i": "<i", "s": "<h", "S": "<H", "I": "<I"}[hp_type]
        aux += b"HP" + hp_type.encode() + struct.pack(fmt, hp)
    if sa is not None:
        aux += b"SAZ" + sa.encode() + b"\0"
    aux += extra_aux
    name = name + b"\0"
    if end is None:
        end = pos + 1
    body = struct.pack("<iiBBHHHIiii", tid, pos, len(name), mapq, reg2bin(max(pos, 0), max(end, pos + 1)), len(cig), flag,
                       l_seq, -1, -1, 0)
    body += name + cig.astype("<u4").tobytes() + aux
    return struct.pack("<I", len(body)) + body


def write_bam(path, ref_names, ref_lens, records, header_text=None):
    """records: iterable of bytes from encode_record, in file order."""
    if header_text is None:
        header_text = "@HD\tVN:1.6\tSO:coordinate\n" + "".join(f"@SQ\tSN:{n}\tLN:{l}\n" for n, l in zip(ref_names, ref_lens))
    ht = header_text.encode()
    head = b"BAM\1" + struct.pack("<I", len(ht)) + ht + struct.pack("<I", len(ref_names))
    for n, l in zip(ref_names, ref_lens):
        nb = n.encode() + b"\0"
        head += struct.pack("<I", len(nb)) + nb + struct.pack("<I", int(l))
    with open(path, "wb") as f:
        buf = bytearray(head)
        for r in records:
            buf += r
            while len(buf) >= 60000:
                f.write(_bgzf_block(bytes(buf[:60000])))
                del buf[:60000]
        if buf:
            f.write(_bgzf_block(bytes(buf)))
        f.write(_EOF)


def reads_to_bam(path, ref_names, ref_lens, reads, rng=None, sa_for_flags=True, hp_type="C"):
    """Write an SoA read set as a BAM. Reads flagged accidental-2D get an SA tag that the host must
    classify as 2D (opposite strand, overlapping); a share of the others get SA tags that must NOT."""
    rng = rng or np.random.default_rng(0)
    recs = []
    for i in range(len(reads.contig)):
        a, b = int(reads.cigar_off[i]), int(reads.cigar_off[i + 1])
        cig = reads.cigar[a:b]
        pos, end = int(reads.ref_start[i]), int(reads.ref_end[i])
        rev = bool(rng.integers(0, 2))
        flag = 0x10 if rev else 0
        sa = None
        if sa_for_flags:
            if reads.flags[i] & 1:
                mid = (pos + end) // 2 + 1
                sa = f"{ref_names[int(reads.contig[i])]},{mid},{'+' if rev else '-'},{max(end - mid, 1)}M10S,60,0;"
            else:
                u = rng.random()
                if u < 0.03:      # same strand
                    sa = f"{ref_names[int(reads.contig[i])]},{pos + 1},{'-' if rev else '+'},50M,60,0;"
                elif u < 0.06:    # two entries
                    sa = f"chr1,{pos + 1},{'+' if rev else '-'},50M,60,0;chr2,5,+,10M,1,0;"
                elif u < 0.09:    # opposite strand but no overlap (starts at end, 1-based POS used as is)
                    sa = f"chrZ,{end},{'+' if rev else '-'},50M,60,0;"
        hp = None if reads.hp[i] == 0xFF else int(reads.hp[i])
        recs.append(encode_record(int(reads.contig[i]), pos, int(reads.mapq[i]), flag, cig, name=f"r{i}".encode(), hp=hp,
                                  hp_type=hp_type, sa=sa, end=end))
    write_bam(path, ref_names, ref_lens, recs)


def index_bam(path: str, meta: bool = False) -> str:
    """Pure-Python BAI builder (SAM spec 5.2) for coordinate-sorted BAMs written by this module or by
    synth.write_bam: bins with merged chunks, 16 kb linear index. meta=True adds what htslib writes on
    top: the metadata pseudo-bin 37450 of every populated reference (its first and last virtual offset,
    mapped / unmapped counts) and the n_no_coor trailer. Returns the .bai path."""
    data = open(path, "rb").read()
    # pass 1: BGZF blocks -> (compressed offset, inflated bytes)
    blocks, off = [], 0
    while off < len(data):
        xlen = struct.unpack_from("<H", data, off + 10)[0]
        bsize = None
        p = off + 12
        while p < off + 12 + xlen:
            si1, si2, slen = data[p], data[p + 1], struct.unpack_from("<H", data, p + 2)[0]
            if si1 == 66 and si2 == 67:
                bsize = struct.unpack_from("<H", data, p + 4)[0] + 1
            p += 4 + slen
        raw = zlib.decompress(data[off + 12 + xlen: off + bsize - 8], -15) if bsize > 12 + xlen + 8 else b""
        blocks.append((off, raw))
        off += bsize
    stream = b"".join(r for _, r in blocks)
    starts, acc = [], 0
    for coff, raw in blocks:
        starts.append((acc, coff, len(raw)))
        acc += len(raw)

    def voffset(pos):  # stream position -> virtual offset (first block that contains it)
        import bisect
        i = bisect.bisect_right([s for s, _, _ in starts], pos) - 1
        while i + 1 < len(starts) and pos >= starts[i][0] + starts[i][2]:
            i += 1
        s, coff, _ = starts[i]
        return (coff << 16) | (pos - s)

    p = 4
    l_text = struct.unpack_from("<I", stream, p)[0]; p += 4 + l_text
    n_ref = struct.unpack_from("<I", stream, p)[0]; p += 4
    for _ in range(n_ref):
        l_name = struct.unpack_from("<I", stream, p)[0]; p += 4 + l_name + 4
    bins = [dict() for _ in range(n_ref)]
    linear = [dict() for _ in range(n_ref)]
    span = [None] * n_ref            # [first v0, last v1, mapped, unmapped] per reference
    n_no_coor = 0
    while p + 4 <= len(stream):
        bs = struct.unpack_from("<I", stream, p)[0]
        tid, pos, l_name, mapq, _bin, n_cig, flag, l_seq = struct.unpack_from("<iiBBHHHI", stream, p + 4)
        cig = np.frombuffer(stream, dtype="<u4", count=n_cig, offset=p + 4 + 32 + l_name)
        rlen = int((cig >> 4)[np.isin(cig & 15, [0, 2, 3, 7, 8])].sum()) if not (flag & 4) else 0
        # CG long cigar: reference length is in the second op (N)
        if n_cig == 2 and (int(cig[0]) & 15) == 4 and (int(cig[1]) & 15) == 3:
            rlen = int(cig[1]) >> 4
        end = pos + max(rlen, 1)
        v0, v1 = voffset(p), voffset(p + 4 + bs)
        if tid >= 0:
            b = reg2bin(pos, end)
            ch = bins[tid].setdefault(b, [])
            if ch and ch[-1][1] == v0:
                ch[-1][1] = v1
            else:
                ch.append([v0, v1])
            for w in range(pos >> 14, ((end - 1) >> 14) + 1):
                if w not in linear[tid]:
                    linear[tid][w] = v0
            s = span[tid] = span[tid] or [v0, v1, 0, 0]
            s[1] = v1
            s[3 if flag & 4 else 2] += 1
        else:
            n_no_coor += 1
        p += 4 + bs
    out = bytearray(b"BAI\1" + struct.pack("<i", n_ref))
    for t in range(n_ref):
        has_meta = meta and span[t] is not None
        out += struct.pack("<i", len(bins[t]) + has_meta)
        for b, chunks in bins[t].items():
            out += struct.pack("<Ii", b, len(chunks))
            for v0, v1 in chunks:
                out += struct.pack("<QQ", v0, v1)
        if has_meta:
            out += struct.pack("<IiQQQQ", 37450, 2, *span[t])
        n_intv = (max(linear[t]) + 1) if linear[t] else 0
        out += struct.pack("<i", n_intv)
        last = 0
        for w in range(n_intv):
            last = linear[t].get(w, last)
            out += struct.pack("<Q", last)
    if meta:
        out += struct.pack("<Q", n_no_coor)
    open(path + ".bai", "wb").write(bytes(out))
    return path + ".bai"
