"""god-aligner without a device: the Python specification against hand-derived records, and the native
BGZF writer + BAI builder (mg_bam_write_sorted) against the specification on synthetic sorted records."""
import gzip
import os
import random
import struct

import pytest

from mitty_b200.simulation.readgenerate import ReadInfo, parse_qname
from tests import bam_spec as S

CONTIGS = [('1', 20000), ('X', 300000), ('virus', 9000)]


def _pair_records():
  # a read inside a long insertion ('>0:2I', reference test_rpc.py:176-180) and a strand-1 mate with X and D
  # carrying corrupted qualities
  name = b'T:0:0:1|1|0|0|8|2|>0:2I|+3|1|12|2|1X1D1=|0,-1'
  infos = parse_qname(name.decode())
  r1 = S.encode_record(name, b'AC', b'IJ', infos[0], infos[1], 0, 0, 'T')
  r2 = S.encode_record(name, b'GT', b'#~', infos[1], infos[0], 1, 0, 'T')
  return name, r1, r2


def test_spec_insertion_read_by_hand():
  name, r1, _ = _pair_records()
  l_name = len(name) + 1
  assert r1[:4] == struct.pack('<i', len(r1) - 4)
  # refID 0, POS 7 (qname pos 8 - 1), l_read_name, MAPQ 60, bin 4681 (0x1249: a zero-length alignment counts as
  # one base), 1 CIGAR op, FLAG 0x63 (paired, proper, first, mate reverse), l_seq 2, mate 0 / 11, TLEN +7 (7..14)
  assert r1[4:36] == (bytes.fromhex('00000000' '07000000') + bytes([l_name, 0x3c]) + bytes.fromhex('4912' '0100' '6300' '02000000' '00000000'
                                                                                                       '0b000000' '07000000'))
  p = 36 + l_name
  assert r1[36:p] == name + b'\0'
  assert r1[p:p + 4] == bytes.fromhex('21000000')             # 2I
  assert r1[p + 4:p + 5] == bytes([0x12])                      # A=1, C=2
  assert r1[p + 5:p + 7] == bytes([40, 41])                    # 'I' - 33, 'J' - 33
  assert r1[p + 7:] == b'RGZT\0'


def test_spec_reverse_read_with_x_and_d_by_hand():
  name, _, r2 = _pair_records()
  l_name = len(name) + 1
  # POS 11, bin 4681 over [11, 14), 3 ops, FLAG 0x93 (paired, proper, reverse, second), mate at 7, TLEN -7
  assert r2[4:36] == (bytes.fromhex('00000000' '0b000000') + bytes([l_name, 0x3c]) + bytes.fromhex('4912' '0300' '9300' '02000000' '00000000'
                                                                                                       '07000000' 'f9ffffff'))
  p = 36 + l_name
  assert r2[p:p + 12] == bytes.fromhex('18000000' '12000000' '17000000')   # 1X 1D 1=
  # 'GT' as read on strand 1: reverse 'TG', complement 'AC' -> 0x12; qualities '#~' reversed -> 93, 2
  assert r2[p + 12:p + 13] == bytes([0x12])
  assert r2[p + 13:p + 15] == bytes([93, 2])


def test_spec_single_end_bin_crossing_lower_case_by_hand():
  name = b'T:0:0:2|1|0|0|16381|10|10=||1|16400|10|10=|'
  info = parse_qname(name.decode())[0]
  r = S.encode_record(name, b'acgtNacgtN', b'IIIIIIIIII', info, None, 0, 0, 'T')
  # POS 16380, [16380, 16390) crosses the 16 kb boundary: bin 585 (0x249); FLAG 0, mate -1 / -1, TLEN 0
  assert r[4:36] == (bytes.fromhex('00000000' 'fc3f0000') + bytes([len(name) + 1, 0x3c]) + bytes.fromhex('4902' '0100' '0000' '0a000000'
                                                                                                            'ffffffff' 'ffffffff' '00000000'))
  p = 36 + len(name) + 1 + 4
  assert r[p:p + 5] == bytes.fromhex('1248f1248f')             # lower case encodes as upper case, N = 15


def test_spec_sort_is_stable_and_template_ordered():
  q = b'@T:0:0:{}|1|0|{}|100|2|2=||{}|100|2|2=|\nAC\n+\nII\n'
  fq1 = q.replace(b'{}', b'1', 1).replace(b'{}', b'1', 1).replace(b'{}', b'0', 1) + q.replace(b'{}', b'2', 1).replace(b'{}', b'0', 1).replace(b'{}', b'0', 1)
  _, recs = S.records(CONTIGS, fq1)
  # same pos: the forward read (template 2) sorts before the reverse one (template 1)
  assert [r[36:43] for r in recs] == [b'T:0:0:2', b'T:0:0:1']


def _synthetic(n=3000, seed=5):
  rng = random.Random(seed)
  recs = []
  for i in range(n):
    rid = rng.choice([0, 1, 1, 2])
    ln = CONTIGS[rid][1]
    cig = rng.choice(['100=', '50=3D50=', '20=1X79=', '40=5I55=', '100I'])
    pos = rng.randrange(1, ln - 200)
    strand = rng.randrange(2)
    info = ReadInfo('T', 'T:0:0:%d' % i, CONTIGS[rid][0], 0, strand, pos, 100, cig, None, [])
    seq = bytes(rng.choice(b'ACGTNacgtRY') for _ in range(100))
    qual = bytes(rng.randrange(35, 75) for _ in range(100))
    name = ('T:0:0:%d|%s|0|%d|%d|100|%s|' % (i, CONTIGS[rid][0], strand, pos, cig)).encode()
    recs.append(((rid, pos - 1, strand), i, S.encode_record(name, seq, qual, info, None, 0, rid, 'T')))
  recs.sort(key=lambda r: (r[0], r[1]))
  return [r[2] for r in recs]


@pytest.fixture(scope='module')
def synthetic():
  return _synthetic()


@pytest.mark.parametrize('level,threads', [(6, 1), (6, 4), (1, 3), (0, 2)])
def test_native_writer_matches_spec(tmp_path, synthetic, level, threads):
  from mitty_b200.engine import write_sorted_bam
  recs = b''.join(synthetic)
  bam, bai = str(tmp_path / 'x.bam'), str(tmp_path / 'x.bam.bai')
  text = S.header_text(CONTIGS, 'T')
  assert write_sorted_bam(bam, bai, CONTIGS, text, recs, level=level, threads=threads) == len(synthetic)
  data = open(bam, 'rb').read()
  ms = S.members(data)                                       # framing, BSIZE <= 64 KiB, CRC32, ISIZE of every member
  assert len(ms) > 10 and data[-28:] == S.EOF_BLOCK
  assert gzip.decompress(data) == S.header_bytes(CONTIGS, 'T') + recs
  assert S.decompress(data) == S.header_bytes(CONTIGS, 'T') + recs
  assert open(bai, 'rb').read() == S.build_bai(data, len(CONTIGS))


def test_native_writer_does_not_depend_on_threads(tmp_path, synthetic):
  from mitty_b200.engine import write_sorted_bam
  recs = b''.join(synthetic)
  out = []
  for t in (1, 2, 7):
    p = str(tmp_path / ('t%d.bam' % t))
    write_sorted_bam(p, p + '.bai', CONTIGS, S.header_text(CONTIGS, 'T'), recs, level=6, threads=t)
    out.append((open(p, 'rb').read(), open(p + '.bai', 'rb').read()))
  assert out[0] == out[1] == out[2]


def test_native_writer_without_records_and_without_index(tmp_path):
  from mitty_b200.engine import write_sorted_bam
  p = str(tmp_path / 'e.bam')
  assert write_sorted_bam(p, None, CONTIGS, S.header_text(CONTIGS, 'T'), b'') == 0
  data = open(p, 'rb').read()
  assert S.decompress(data) == S.header_bytes(CONTIGS, 'T') and not os.path.exists(p + '.bai')
  # a truncated record stream is an error and leaves no file behind
  with pytest.raises(ValueError):
    write_sorted_bam(p, p + '.bai', CONTIGS, S.header_text(CONTIGS, 'T'), _synthetic(3)[0][:-3])
  assert not os.path.exists(p) and not os.path.exists(p + '.bai')


def test_index_query_finds_every_overlapping_record(tmp_path, synthetic):
  from mitty_b200.engine import write_sorted_bam
  p = str(tmp_path / 'q.bam')
  write_sorted_bam(p, p + '.bai', CONTIGS, S.header_text(CONTIGS, 'T'), b''.join(synthetic), level=1, threads=2)
  rng = random.Random(11)
  regions = []
  for _ in range(200):
    ref = rng.randrange(len(CONTIGS))
    beg = rng.randrange(CONTIGS[ref][1] - 10)
    regions.append((ref, beg, min(CONTIGS[ref][1], beg + rng.choice([1, 50, 1000, 20000, 100000]))))
  S.check_queries(open(p, 'rb').read(), open(p + '.bai', 'rb').read(), regions)


# ---- block, record-size and bin edges of the writer -------------------------------------------------

EDGE_CONTIGS = [('1', 20000), ('big', 3 * (1 << 26) + 12345), ('empty', 5000), ('last', 1 << 27)]


def _reads(rng, chrom, n, length, L=60):
  """n single-end templates of L bases at random positions of chrom, in coordinate order."""
  return sorted(((chrom, [(rng.randrange(2), rng.randrange(1, length - L), '%d=' % L, bytes(rng.choice(b'ACGT') for _ in range(L)), b'I' * L)])
                 for _ in range(n)), key=lambda t: t[1][0][1::-1])


def _stream(templates, pad=None):
  """-> (header + records, records) of the spec for single-end templates."""
  fq1, _ = S.fastq(templates, sample='T', pad=pad)
  _, recs = S.records(EDGE_CONTIGS, fq1)
  return S.header_bytes(EDGE_CONTIGS, 'T') + b''.join(recs), recs


def _bin_edge_templates(rng):
  out = []
  for ref in (1, 3):
    chrom, length = EDGE_CONTIGS[ref]
    for beg, sp in S.bin_edge_spans(length):
      pos, cig, rlen = S.read_layout(beg, sp)
      out.append((chrom, [(rng.randrange(2), pos, cig, bytes(rng.choice(b'ACGT') for _ in range(rlen)), b'5' * rlen)]))
  return out


def _padded_to(templates, target):
  """Pads the names of the first templates (in coordinate order) so that a record ends exactly at
  uncompressed offset ``target``.  -> pad"""
  raw, recs = _stream(templates)
  u = len(raw) - sum(len(r) for r in recs)
  ends = []
  for r in recs:
    u += len(r)
    ends.append(u)
  short = max(e for e in ends if e <= target)       # the last record end at or before target, moved up to it
  need, pad = target - short, [0] * len(templates)
  for t in range(len(templates)):
    pad[t] = min(need, 150)
    need -= pad[t]
  assert need == 0
  return pad


def _edge_case(case):
  rng = random.Random(case)
  if case == 'bins_0_to_72':
    t = _bin_edge_templates(rng) + _reads(rng, '1', 300, 20000)
    return t, None
  if case == 'record_over_64k':
    L = 100000
    big = ('big', [(1, 5000, '%d=' % L, bytes(rng.choice(b'ACGTN') for _ in range(L)), bytes(rng.randrange(33, 75) for _ in range(L)))])
    return _reads(rng, 'big', 400, 20000) + [big] + _reads(rng, 'big', 200, 200000), None
  t = _reads(rng, '1', 1500, 20000)
  raw, _ = _stream(t)
  if case == 'record_ends_on_block':
    return t, _padded_to(t, S.BLOCK)
  assert case == 'stream_is_whole_blocks'
  return t, _padded_to(t, (len(raw) // S.BLOCK + 1) * S.BLOCK)


@pytest.mark.parametrize('case', ['bins_0_to_72', 'record_ends_on_block', 'stream_is_whole_blocks', 'record_over_64k'])
def test_native_writer_block_record_and_bin_edges(tmp_path, case):
  """The native writer and index against the specification where blocks, records and bins meet their edges;
  each case asserts that its records reach the edge it is named after."""
  from mitty_b200.engine import write_sorted_bam
  templates, pad = _edge_case(case)
  raw, recs = _stream(templates, pad)
  ends, u = set(), len(raw) - sum(len(r) for r in recs)
  for r in recs:
    u += len(r)
    ends.add(u)
  bins = {struct.unpack_from('<H', r, 14)[0] for r in recs}
  if case == 'bins_0_to_72':
    assert 0 in bins and bins & set(range(1, 9)) and bins & set(range(9, 73)) and bins & set(range(73, 585)), sorted(bins)[:20]
  elif case == 'record_ends_on_block':
    assert S.BLOCK in ends and len(raw) > 2 * S.BLOCK
  elif case == 'stream_is_whole_blocks':
    assert len(raw) % S.BLOCK == 0 and len(raw) // S.BLOCK >= 2
  else:
    assert max(len(r) for r in recs) > 1 << 16
  p = str(tmp_path / 'e.bam')
  assert write_sorted_bam(p, p + '.bai', EDGE_CONTIGS, S.header_text(EDGE_CONTIGS, 'T'), b''.join(recs), level=1, threads=3) == len(recs)
  data, bai = open(p, 'rb').read(), open(p + '.bai', 'rb').read()
  assert S.decompress(data) == raw
  assert bai == S.build_bai(data, len(EDGE_CONTIGS))
  if case == 'stream_is_whole_blocks':
    assert [len(m) for _, m in S.members(data)] == [S.BLOCK] * (len(raw) // S.BLOCK) + [0]
  if case == 'bins_0_to_72':
    S.check_queries(data, bai, S.edge_queries(1, EDGE_CONTIGS[1][1]) + S.edge_queries(3, EDGE_CONTIGS[3][1]) + [(2, 0, 5000)])


def test_writer_rejects_contigs_bam_cannot_address(tmp_path):
  """BAM keeps a contig's length, POS, PNEXT and TLEN in int32: a contig of 2^31 bases or more is an error
  naming it, raised before any file exists; 2^31 - 1 bases are written."""
  from mitty_b200.engine import write_sorted_bam
  p = str(tmp_path / 'x.bam')
  for length in (1 << 31, 1 << 40):
    contigs = [('1', 100), ('huge', length)]
    with pytest.raises(ValueError, match='huge'):
      write_sorted_bam(p, p + '.bai', contigs, 'x', b'')
    assert os.listdir(str(tmp_path)) == []
  contigs = [('1', 100), ('huge', (1 << 31) - 1)]
  assert write_sorted_bam(p, None, contigs, S.header_text(contigs, 'T'), b'') == 0
  assert S.decompress(open(p, 'rb').read()) == S.header_bytes(contigs, 'T')


def test_spec_bin_past_2_29_keeps_its_low_16_bits():
  """Past 2^29 the SAM spec's bin no longer fits the record's 16-bit field (from 4681 + 997 048 320 >> 14):
  the record keeps its low 16 bits, as htslib's uint16_t field does."""
  for pos0, sp, full in ((1 << 29, 10, 4681 + (1 << 15)), (997048320 - 1, 1, 65535), (997048320, 1, 65536),
                         ((1 << 31) - 2, 1, 4681 + ((1 << 31) - 2 >> 14)), ((1 << 30) + 3, 1 << 16, 585 + (1 << 13))):
    assert S.reg2bin(pos0, pos0 + sp) == full
    name = b'T:0:0:1|h|0|0|%d|%d|%d=|' % (pos0 + 1, sp, sp)
    r = S.encode_record(name, b'A' * sp, b'I' * sp, parse_qname(name.decode())[0], None, 0, 0, 'T')
    assert struct.unpack_from('<i', r, 8)[0] == pos0
    assert struct.unpack_from('<H', r, 14)[0] == full & 0xFFFF
