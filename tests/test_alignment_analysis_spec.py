"""alignment-analysis without a device: the specification (tests/alignment_analysis_spec.py) against hand-computed
matrices and counters for every rule and error, and the CSV writer's layout and atomic write."""
import os
import struct

import numpy as np
import pytest

from tests import alignment_analysis_spec as A

NAMES = [b'c', b'cc', b'd']
CONTIGS = [(n.decode(), 100000) for n in NAMES]


def R(reads=((0, 101, 4, '4=', ''),), chrom=b'c', flag=0, ref=0, pos=100, mapq=60, cigar=((4, 7),)):
  """A record of a read whose truth is `reads` (strand, pos, rlen, CIGAR, v_list per read of the template)."""
  return A.record(name=A.qname(chrom, reads), flag=flag, ref=ref, pos=pos, mapq=mapq, cigar=cigar, seq=b'ACGT', qual=[30] * 4)


S, H, I, P, EQ, M, D = 4, 5, 1, 6, 7, 0, 2
PAIR = ((0, 101, 4, '4=', ''), (1, 201, 4, '4=', '3'))

# (record, expected column offset d (or 'wc' / 'un' / None for skipped), mapq, v_list)
CASES = [
  (R(), 0, 60, []),                                                              # 0 truth alignment
  (R(pos=102, cigar=((2, S), (2, EQ))), 0, 60, []),                              # 1 leading soft clip moves POS
  (R(pos=103, cigar=((3, H), (4, EQ))), 0, 60, []),                              # 2 leading hard clip
  (R(pos=105, cigar=((2, H), (3, S), (4, EQ))), 0, 60, []),                      # 3 H + S
  (R(pos=101, cigar=((1, I), (3, EQ))), 0, 60, []),                              # 4 leading insertion on the aligned side
  (R(pos=102, cigar=((1, S), (1, P), (1, S), (2, EQ))), 0, 60, []),              # 5 P inside the leading run is skipped
  (R(reads=((0, 101, 4, '2I2=', ''),), pos=100, cigar=((2, I), (2, EQ))), 0, 60, []),   # 6 truth with a leading kI
  (R(reads=((0, 101, 4, '>3:4I', '4'),), pos=100, cigar=((4, I),)), 0, 60, [4]),       # 7 '>p:nI' read inside an insertion
  (R(pos=103, mapq=0), 3, 0, []),                                                # 8 d = +3
  (R(pos=93, mapq=255), -7, 255, []),                                            # 9 d = -7, clamped at max_d = 5
  (R(ref=-1, pos=-1, cigar=()), 'un', 60, []),                                   # 10 refID -1 without 0x4
  (R(flag=0x4), 'un', 60, []),                                                   # 11 0x4 with a valid refID
  (R(ref=1), 'wc', 60, []),                                                      # 12 'c' is a prefix of header name 'cc'
  (R(chrom=b'cc', ref=0), 'wc', 60, []),                                         # 13 'cc' against header name 'c'
  (R(flag=0x100, ref=7), None, 0, []),                                           # 14 secondary: skipped, refID not even checked
  (R(flag=0x800, chrom=b'not|mitty'), None, 0, []),                              # 15 supplementary: skipped
  (R(reads=PAIR, flag=0x93, pos=200, mapq=30), 0, 30, [3]),                               # 16 read 2 of a pair (reverse, as in the qname)
  (R(reads=PAIR, flag=0x0), 0, 60, []),                                          # 17 paired qname on an unpaired record: read 1's fields
  (R(flag=0x600, reads=((0, 101, 4, '4=', '-5,,-2,0,2,7'),)), 0, 60, [-5, -2, 0, 2, 7]),   # 18 QC-fail + duplicate analysed
  (R(flag=0x10), 0, 60, []),                                                     # 19 strand mismatch
]


def test_hand_computed_rules():
  recs = [r for r, _, _, _ in CASES]
  got = A.analyse(recs, NAMES, max_d=5, max_size=2)
  C = 13
  mq, vs = np.zeros((256, C), dtype=np.uint64), np.zeros((8, C), dtype=np.uint64)
  col = {'un': 12, 'wc': 11}
  for _, d, q, vl in CASES:
    if d is None:
      continue
    c = col[d] if d in col else min(max(d, -5), 5) + 5
    mq[q, c] += 1
    for v in vl:                                  # rows: del>2, -2 .. 2, ins>2, none
      vs[{-5: 0, -2: 1, 0: 3, 2: 5, 3: 6, 4: 6, 7: 6}[v], c] += 1
    if not vl:
      vs[7, c] += 1
  assert np.array_equal(got['mq'], mq) and np.array_equal(got['vsize'], vs)
  assert got['mq'][60, 5] == 11 and got['mq'][0, 8] == 1 and got['mq'][255, 0] == 1
  assert {k: got[k] for k in A.COUNTERS} == {'records': 20, 'analysed': 18, 'skipped': 2, 'unmapped': 2, 'wrong_chrom': 2, 'exact': 12,
                                             'clamped': 1, 'strand_mismatch': 1, 'no_variant_reads': 15, 'variant_entries': 7}


def test_max_d_zero_and_max_size_zero():
  recs = [R(), R(pos=103), R(pos=97), R(ref=1), R(flag=4, reads=((0, 101, 4, '4=', '-1,0,1'),))]
  got = A.analyse(recs, NAMES, max_d=0, max_size=0)
  assert got['mq'].shape == (256, 3) and got['vsize'].shape == (4, 3)
  assert got['mq'][60].tolist() == [3, 1, 1]
  assert got['vsize'].tolist() == [[0, 0, 1], [0, 0, 1], [0, 0, 1], [3, 1, 0]]
  assert (got['exact'], got['clamped']) == (1, 2)


def _one(rec, names=NAMES):
  return A.analyse([R(), rec], names)


ERRORS = {
  'refid_high': (R(ref=3), 'refID out of range'),
  'refid_low': (R(ref=-2), 'refID out of range'),
  'refid_before_qname': (A.record(name=b'junk', ref=9), 'refID out of range'),
  'few_fields': (A.record(name=b'a|b|c|0|1|4|4='), 'not a Mitty qname'),
  'no_name': (A.record(name=b''), 'not a Mitty qname'),
  'strand_2': (R(reads=((2, 101, 4, '4=', ''),)), 'not a Mitty qname'),
  'strand_text': (R(reads=(('x', 101, 4, '4=', ''),)), 'not a Mitty qname'),
  'pos_plus': (R(reads=((0, '+101', 4, '4=', ''),)), 'not a Mitty qname'),
  'pos_huge': (R(reads=((0, 2 ** 40 + 1, 4, '4=', ''),)), 'not a Mitty qname'),
  'cigar_op': (R(reads=((0, 101, 4, '4Q', ''),)), 'not a Mitty qname'),
  'cigar_empty': (R(reads=((0, 101, 4, '', ''),)), 'not a Mitty qname'),
  'cigar_no_count': (R(reads=((0, 101, 4, '=', ''),)), 'not a Mitty qname'),
  'cigar_special_offset': (R(reads=((0, 101, 4, '>x:4I', ''),)), 'not a Mitty qname'),
  'cigar_special_no_colon': (R(reads=((0, 101, 4, '>4I', ''),)), 'not a Mitty qname'),
  'vlist_entry': (R(reads=((0, 101, 4, '4=', '1,a'),)), 'not a Mitty qname'),
  'mate_missing': (R(flag=0x81), 'no read for this mate'),
  'mate_missing_short': (A.record(name=b'a|b|c|0|1', flag=0x81), 'not a Mitty qname'),
}


@pytest.mark.parametrize('case', sorted(ERRORS))
def test_errors(case):
  rec, what = ERRORS[case]
  with pytest.raises(A.SpecError) as e:
    _one(rec)
  assert (e.value.kind, e.value.where) == ('record', 1) and str(e.value).endswith(what)


def test_unmapped_and_skipped_records_are_still_checked_or_not():
  """An unmapped record's qname must still be Mitty's; a skipped record is not looked at."""
  with pytest.raises(A.SpecError, match='record 1: not a Mitty qname'):
    _one(A.record(name=b'x', flag=4, ref=-1))
  assert _one(A.record(name=b'x', flag=0x904, ref=-5))['skipped'] == 1


def test_first_bad_record_in_stream_order(tmp_path):
  """A qname error before a framing error is reported, and a framing error before a qname error."""
  good, bad = R(), A.record(name=b'x')
  raw = A.header(CONTIGS) + good * 3 + bad + good
  cut = A.header(CONTIGS) + good * 2
  with pytest.raises(A.SpecError, match='record 3: not a Mitty qname'):
    A.analysis(A.bgzf(raw + bytes(good[:10]), cuts=300))
  with pytest.raises(A.SpecError, match='record 2: cut off'):
    A.analysis(A.bgzf(cut + bytes(good[:10]) + bad, cuts=300))
  data = A.bgzf(raw, cuts=50)
  offs = [o for o, _ in A.members(data)]
  m = (len(A.header(CONTIGS)) + 3 * len(good) + len(bad)) // 50 + 1   # a member after record 3
  b = bytearray(data)
  b[offs[m + 1] - 8] ^= 1
  with pytest.raises(A.SpecError, match='record 3: not a Mitty qname'):
    A.analysis(bytes(b))
  b = bytearray(data)
  b[offs[1] - 8] ^= 1                               # a member inside the header
  with pytest.raises(A.SpecError, match='offset 0: CRC32'):
    A.analysis(bytes(b))


def test_header_names_up_to_their_nul():
  raw = A.header(CONTIGS)
  assert A.header_info(raw) == (len(raw), NAMES)
  hand = b'BAM\1' + struct.pack('<ii', 0, 2) + struct.pack('<i', 4) + b'ab\0z' + struct.pack('<ii', 5, 0) + struct.pack('<i', 0)
  assert A.header_info(hand) == (len(hand), [b'ab', b''])         # 'ab' then bytes after its NUL; an empty name


def test_csv_layout_and_atomic_write(tmp_path):
  from mitty_b200.benchmarking.alignment_analysis import read_csv, write_csv
  got = A.analyse([r for r, _, _, _ in CASES], NAMES, max_d=5, max_size=2)
  d = tmp_path / 'out'
  d.mkdir()
  prefix = str(d / 'run')
  umask = os.umask(0o022)
  try:
    paths = write_csv(prefix, got)
  finally:
    os.umask(umask)
  assert paths == (prefix + '.mq.csv', prefix + '.vsize.csv')
  assert sorted(os.listdir(str(d))) == ['run.mq.csv', 'run.vsize.csv']
  assert all(os.stat(p).st_mode & 0o777 == 0o644 for p in paths)
  lines = open(paths[0]).read().splitlines()
  assert lines[0] == 'mq,-5,-4,-3,-2,-1,0,1,2,3,4,5,wrong_chrom,unmapped' and len(lines) == 257
  assert lines[61] == '60,0,0,0,0,0,11,0,0,0,0,0,2,2'
  cols, rows, m = read_csv(paths[0])
  assert rows == [str(q) for q in range(256)] and np.array_equal(m, got['mq'])
  cols, rows, m = read_csv(paths[1])
  assert open(paths[1]).readline().startswith('v_size,-5,')
  assert rows == ['del>2', '-2', '-1', '0', '1', '2', 'ins>2', 'none'] and np.array_equal(m, got['vsize'])
  # a failed write leaves neither the targets nor a temporary file; existing outputs are replaced whole
  import mitty_b200.benchmarking.alignment_analysis as aa
  real, calls = aa._write_atomic, []

  def second_fails(path, text):
    calls.append(path)
    if len(calls) == 2:
      raise OSError('disk full')
    return real(path, text)

  aa._write_atomic = second_fails
  try:
    with pytest.raises(OSError, match='disk full'):
      write_csv(str(d / 'new'), got)
  finally:
    aa._write_atomic = real
  assert sorted(os.listdir(str(d))) == ['run.mq.csv', 'run.vsize.csv']
  write_csv(prefix, A.analyse([R()], NAMES, max_d=0, max_size=0))
  assert read_csv(paths[0])[2].shape == (256, 3) and sorted(os.listdir(str(d))) == ['run.mq.csv', 'run.vsize.csv']


def test_cli_rejects_out_of_range_options(tmp_path):
  from click.testing import CliRunner
  from mitty_b200.cli import cli
  bam = tmp_path / 'x.bam'
  bam.write_bytes(b'')
  for opt in (['--max-d', '10001'], ['--max-size', '-1']):
    res = CliRunner().invoke(cli, ['alignment-analysis', str(bam), str(tmp_path / 'o')] + opt)
    assert res.exit_code == 2 and 'range' in res.output
  assert os.listdir(str(tmp_path)) == ['x.bam']
