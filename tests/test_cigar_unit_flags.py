"""The scan tests both 16-bit units of a word at once from their flag bits (inq_device.cuh, "CIGAR units"): C
(consumes), E (I, D or S), the 2-bit sub field (S, or two payload bits of a long head) and a 12-bit length compared
against minlen in both halves with one subtraction. These cases add what test_cigar_units.py does not run: minlen values
at the edges of that subtraction, long heads whose payload units take every sub value, and a stream whose last read ends
right before the zero padding at the end of a warp tile."""
import numpy as np
import pytest

from oracle.oracle import Reads
from tests.test_cigar_units import check, long_case

MINLENS = (2047, 2048, 4093, 4098)
# I/D/S lengths on both sides of those minlen values, and long heads whose low payload (len & 0x3FFF) and high
# payload (len >> 14) carry each value of the two payload bits that go to the sub field
LENS = (2046, 2047, 2048, 2049, 4092, 4093, 4094, 4096, 4097, 4098, 4099,
        4097 + (1 << 14), 4098 + (2 << 14), 4099 + (3 << 14))
TILE_UNITS = 16384          # the stream is zero-padded to this many units (kTileUnits), 8 warp tiles of 2048


def unit_count(w: np.ndarray) -> np.ndarray:
    """units each BAM word becomes (unit_count in inq_device.cuh)"""
    op, ln = w & 15, (w >> 4).astype(np.int64)
    pieces = (ln + 4094) // 4095
    n = np.where(np.isin(op, [0, 3, 7, 8]), pieces, 0)
    n = np.where(np.isin(op, [1, 4]), np.where(ln < 4095, 1, 3), n)
    n = np.where(op == 2, np.where(ln < 4095, 1, 3 + (np.maximum(ln - 4095, 0) + 4094) // 4095), n)
    return np.where(ln == 0, 0, n)


def with_tail_read(case, tail_residue: int):
    """case plus one last read of 1I fillers and a closing 20I, sized so that the stream ends `tail_residue` units into a
    padding tile (0: exactly at its end, no padding); the zero padding of the stream follows the read. Returns the case
    and the stream's length in units by unit_count"""
    rd = case["reads"]
    used = int(unit_count(rd.cigar.astype(np.int64)).sum())
    fill = (tail_residue - used - 1) % TILE_UNITS + TILE_UNITS
    words = np.concatenate([np.full(fill, (1 << 4) | 1, np.uint32), [np.uint32((20 << 4) | 1)]])
    c, s = int(case["locus_contig"][0]), int(case["locus_start"][0])
    off = np.concatenate([rd.cigar_off, [rd.cigar_off[-1] + len(words)]]).astype(np.uint64)
    reads = Reads(np.append(rd.contig, c), np.append(rd.ref_start, s), np.append(rd.ref_end, s + 1),
                  np.append(rd.mapq, 60), np.append(rd.hp, 1), np.append(rd.flags, 0), off,
                  np.concatenate([rd.cigar, words]).astype(np.uint32))
    return dict(case, reads=reads), used + len(words)


@pytest.fixture(scope="module")
def ctx():
    import inquistr_b200 as q
    c = q.Context(0)
    yield c
    c.close()


def test_unit_count_model():
    w = np.asarray([(4094 << 4) | 0, (4095 << 4) | 0, (4096 << 4) | 3, (4094 << 4) | 2, (4095 << 4) | 2, (8191 << 4) | 2,
                    (4095 << 4) | 1, (5000 << 4) | 4, (7 << 4) | 5, (7 << 4) | 6, (7 << 4) | 9, (0 << 4) | 0], np.uint32)
    assert unit_count(w).tolist() == [1, 1, 2, 1, 3, 5, 3, 3, 0, 0, 0, 0]


@pytest.mark.gpu
@pytest.mark.parametrize("unphased", [False, True])
def test_minlen_edges_and_payload_sub_values(ctx, unphased):
    case = long_case(11, n_lens=LENS)
    ctx.set_loci(case["contig_off"], case["locus_start"], case["locus_end"])
    ctx.clear_reads()
    ctx.push(case["reads"])
    for minlen in MINLENS:
        check(ctx, case, minlen, unphased)


# 16382: the last unit is the high unit of the second-to-last word of lane 31 of a warp tile, the last word is padding;
# 16383: the last unit is the low unit of that lane's last word, its high unit is padding; 1: the last unit opens a
# tile that is padding from there on; 0: no padding. The cases share every unit but the filler's, so the device's tile
# count at 0 and 1 pins unit_count to the encoder: a model that is off in either direction moves one of them across
# the tile edge.
@pytest.mark.gpu
@pytest.mark.parametrize("tail_residue", [16382, 16383, 0, 1])
def test_last_read_before_padding_at_warp_tile_end(ctx, tail_residue):
    case, n_units = with_tail_read(long_case(12, n_reads=100, n_lens=(5, 4095)), tail_residue)
    ctx.set_loci(case["contig_off"], case["locus_start"], case["locus_end"])
    ctx.clear_reads()
    ctx.push(case["reads"])
    for minlen in (5, 19, 20, 4095):
        res = check(ctx, case, minlen, False)
        assert res.stats["n_tiles"] == -(-n_units // TILE_UNITS)
