"""alignment-analysis on the device: every matrix and counter equals the pure-Python specification
(tests/alignment_analysis_spec.py) on god-aligner BAMs (every read scores d = 0), on aligner-like BAMs perturbed
from them, whatever the BGZF layout, chunk size and inflate threads; malformed input raises ValueError naming the
record and leaves nothing behind; the round trip generate-reads -> god-aligner -> alignment-analysis counts every
v_list entry of the FASTQ pair; the command runs on a file and on a FIFO."""
import os
import struct
import threading

import numpy as np
import pytest

from tests import alignment_analysis_spec as A
from tests.test_gpu_read_model import config5_bams, edge_bams  # noqa: F401 (module fixtures: god-aligner BAMs)

pytestmark = pytest.mark.gpu

COUNTERS = A.COUNTERS


@pytest.fixture(scope='module')
def engine():
  from mitty_b200.engine import Engine
  e = Engine(0)
  yield e
  e.close()


def _same(got, want):
  for k in ('mq', 'vsize'):
    assert got[k].dtype == np.uint64 and got[k].shape == want[k].shape and np.array_equal(got[k], want[k]), k
  assert {k: got[k] for k in COUNTERS} == {k: want[k] for k in COUNTERS}


def _check(engine, path, max_d=200, max_size=50, **kw):
  data = open(path, 'rb').read()
  got = engine.alignment_error_counts(path, max_d=max_d, max_size=max_size, **kw)
  _same(got, A.analysis(data, max_d=max_d, max_size=max_size))
  assert got['inflated_bytes'] == sum(len(r) for _, r in A.members(data)) and got['compressed_bytes'] == len(data)
  return got


def _god_bams(edge_bams, config5_bams):  # noqa: F811
  out = {'edge_' + k: v for k, v in edge_bams.items()}
  out.update({'config5_{}_{}'.format(n, 'paired' if p else 'single'): v for (n, p), v in config5_bams.items()})
  return out


@pytest.mark.parametrize('which', ['edge_perfect', 'edge_corrupt', 'config5_normal_paired', 'config5_normal_single', 'config5_tumor_paired',
                                   'config5_tumor_single'])
def test_god_aligner_bams_score_zero(engine, edge_bams, config5_bams, which):  # noqa: F811
  got = _check(engine, _god_bams(edge_bams, config5_bams)[which], threads=4)
  n = got['records']
  assert n > 0 and got['analysed'] == got['exact'] == n and got['strand_mismatch'] == 0
  assert got['mq'][60, 200] == n and got['mq'].sum() == n
  assert got['vsize'][:, 200].sum() == got['variant_entries'] + got['no_variant_reads'] == got['vsize'].sum()
  assert got['variant_entries'] > 0


# ---- aligner-like BAMs perturbed from god-aligner records ------------------------------------------------------

def _with_decoy(raw):
  """The inflated BAM's header with one more contig, 'decoy', and its records."""
  u, names = A.header_info(raw)
  l_text = struct.unpack_from('<i', raw, 4)[0]
  head = raw[:8 + l_text] + struct.pack('<i', len(names) + 1) + raw[12 + l_text:u] + struct.pack('<i', 6) + b'decoy\0' + struct.pack('<i', 1000)
  return head, A.records(raw), len(names) + 1


def _set_cigar(rec, ops):
  l_name, n_cig = rec[12], struct.unpack_from('<H', rec, 16)[0]
  body = bytearray(rec[4:36 + l_name])
  struct.pack_into('<H', body, 12, len(ops))
  new = bytes(body) + b''.join(struct.pack('<I', n << 4 | op) for n, op in ops) + rec[36 + l_name + 4 * n_cig:]
  return struct.pack('<i', len(new)) + new


def _perturbed(path, seed=11):
  """POS shifts within and beyond +/-200 and +/-5, soft and hard clips that move POS (d stays 0), records moved to
  another contig, unmapped records (0x4, and refID -1 without it), secondary and supplementary copies, random MAPQ
  0..255 and flipped strand bits."""
  rng = np.random.RandomState(seed)
  head, recs, n_ref = _with_decoy(b''.join(r for _, r in A.members(open(path, 'rb').read())))
  out = []
  for rec in recs:
    r = bytearray(rec)
    ref, pos = struct.unpack_from('<ii', r, 4)
    flag = struct.unpack_from('<H', r, 18)[0]
    r[13] = int(rng.randint(0, 256))
    what = rng.randint(0, 10)
    if what == 0:
      struct.pack_into('<i', r, 8, pos + int(rng.choice([-1, 1]) * rng.choice([1, 3, 5, 6, 150, 200, 201, 5000])))
    elif what == 1:
      struct.pack_into('<i', r, 4, (ref + 1 + int(rng.randint(n_ref - 1))) % n_ref)
    elif what == 2:
      struct.pack_into('<H', r, 18, flag | 0x4)
    elif what == 3:
      struct.pack_into('<i', r, 4, -1)
    elif what == 4:
      struct.pack_into('<H', r, 18, flag ^ 0x10)
    elif what == 5:
      l_name, n_cig = r[12], struct.unpack_from('<H', r, 16)[0]
      ops = [(x >> 4, x & 15) for x in struct.unpack_from('<%dI' % n_cig, r, 36 + l_name)]
      if ops[0][1] in (7, 8) and ops[0][0] > 1:
        k = int(rng.randint(1, ops[0][0]))
        h = int(rng.randint(0, k + 1))             # k bases clipped: h hard, k - h soft; POS moves by k
        clip = [(n, op) for n, op in ((h, 5), (k - h, 4)) if n]
        struct.pack_into('<i', r, 8, pos + k)
        r = bytearray(_set_cigar(bytes(r), clip + [(ops[0][0] - k, ops[0][1])] + ops[1:]))
    out.append(bytes(r))
    if what in (6, 7):
      c = bytearray(rec)
      struct.pack_into('<H', c, 18, flag | (0x100 if what == 6 else 0x800))
      struct.pack_into('<i', c, 8, pos + int(rng.randint(-10000, 10000)))
      out.append(bytes(c))
  return head + b''.join(out)


@pytest.fixture(scope='module')
def perturbed(tmp_path_factory, config5_bams):  # noqa: F811
  d = tmp_path_factory.mktemp('perturbed')
  out = {}
  for paired in (True, False):
    raw = _perturbed(config5_bams['normal', paired])
    p = str(d / ('p{}.bam'.format(int(paired))))
    open(p, 'wb').write(A.bgzf(raw, cuts=30000))
    out[paired] = (p, raw)
  return out


@pytest.mark.parametrize('paired', [True, False])
@pytest.mark.parametrize('max_d', [0, 5, 200])
@pytest.mark.parametrize('max_size', [0, 50])
def test_perturbed_aligner_bams(engine, perturbed, paired, max_d, max_size):
  got = _check(engine, perturbed[paired][0], max_d=max_d, max_size=max_size, threads=3)
  assert all(got[k] > 0 for k in ('skipped', 'unmapped', 'wrong_chrom', 'strand_mismatch', 'exact', 'no_variant_reads', 'variant_entries'))
  assert got['clamped'] > 0
  assert np.count_nonzero(got['mq'].sum(axis=1)) > 200                       # random MAPQ reaches most rows


def test_layout_chunks_threads_do_not_matter(engine, perturbed, tmp_path):
  """Random member cuts, the header's name list cut into one-byte members, records larger than the 128 KiB least
  chunk (so that a chunk holds one record), and 1 / 3 / 16 threads."""
  raw = perturbed[True][1]
  u, names = A.header_info(raw)
  big = [A.record(name=A.qname(names[0], ((0, 1001 + i, 70000, '70000=', '1,-2'),)), pos=1000 + i, cigar=((70000, 7),), seq=b'A' * 70000,
                  qual=[30] * 70000) for i in range(3)]
  recs = A.records(raw)
  raw = raw[:u] + big[0] + b''.join(recs[:500]) + big[1] + b''.join(recs[500:]) + big[2]
  rng = np.random.RandomState(8)
  cuts = [1] * u + [int(x) for x in rng.randint(1, 30000, 400)]
  total = 0
  for i, c in enumerate(cuts):
    total += c
    if total >= len(raw):
      cuts = cuts[:i]
      break
  data = A.bgzf(raw, cuts=cuts, level=lambda k: int(rng.randint(0, 10)), empty_every=7)
  p = str(tmp_path / 'l.bam')
  open(p, 'wb').write(data)
  for threads in (1, 3, 16):
    for chunk in (1, 1 << 20, 64 << 20):
      got = _check(engine, p, max_d=5, max_size=3, threads=threads, chunk_bytes=chunk)
      if chunk == 1:
        assert got['chunks'] >= len(raw) // (1 << 17)
  assert got['records'] == len(recs) + 3 and got['exact'] > 0


# ---- errors ------------------------------------------------------------------------------------------------------

def _error_input(edge_bams, case):  # noqa: F811
  """-> (BGZF bytes, 'record' | 'offset', where) of one malformed input built from the perfect edge BAM."""
  raw = b''.join(r for _, r in A.members(open(edge_bams['perfect'], 'rb').read()))
  u, names = A.header_info(raw)
  recs = A.records(raw)
  k = 300
  r = bytearray(recs[k])
  l_name = r[12]
  if case == 'cigar_overrun':
    struct.pack_into('<H', r, 16, 0xFFFF)
  elif case == 'seq_overrun':
    struct.pack_into('<i', r, 20, 2 ** 31 - 1)
  elif case == 'block_size':
    struct.pack_into('<i', r, 0, 31)
  elif case == 'refid':
    struct.pack_into('<i', r, 4, len(names))
  elif case in ('qname', 'mate'):
    name = bytes(r[36:36 + l_name - 1])
    if case == 'qname':
      name = name.replace(b'|', b'/', 4)
    else:
      name = b'|'.join(name.split(b'|')[:8])
      struct.pack_into('<H', r, 18, 0x91)
    n_cig = struct.unpack_from('<H', r, 16)[0]
    body = bytearray(r[4:36])
    body[8] = len(name) + 1
    r = bytearray(struct.pack('<i', 32 + len(name) + 1 + len(r) - 36 - l_name) + bytes(body) + name + b'\0' + bytes(r[36 + l_name:]))
    assert struct.unpack_from('<H', r, 16)[0] == n_cig
  bad = raw[:u] + b''.join(recs[:k]) + bytes(r) + b''.join(recs[k + 1:])
  if case == 'cut':
    return A.bgzf(raw[:u] + b''.join(recs[:k]) + recs[k][:50], cuts=7000), 'record', k
  if case == 'crc':
    data = A.bgzf(raw, cuts=7000)
    offs = [o for o, _ in A.members(data)]
    b = bytearray(data)
    b[offs[4] - 8] ^= 1
    return bytes(b), 'offset', offs[3]
  return A.bgzf(bad, cuts=7000), 'record', k


ERROR_CASES = {'cigar_overrun': 'CIGAR overruns block_size', 'seq_overrun': 'SEQ overruns block_size', 'block_size': 'block_size < 32',
               'cut': 'the file ends inside the record', 'crc': 'CRC32 mismatch', 'refid': 'refID out of range',
               'qname': 'not a Mitty qname', 'mate': 'no read for this mate in the qname'}


@pytest.mark.parametrize('case', sorted(ERROR_CASES))
def test_errors_name_the_record_and_leave_nothing(tmp_path, edge_bams, case):  # noqa: F811
  from mitty_b200.benchmarking.alignment_analysis import process_bam
  data, kind, where = _error_input(edge_bams, case)
  with pytest.raises(A.SpecError) as e:
    A.analysis(data)
  assert (e.value.kind, e.value.where) == (kind, where)
  d = tmp_path / 'e'
  d.mkdir()
  bam = str(d / 'bad.bam')
  open(bam, 'wb').write(data)
  for chunk in (1 << 17, 64 << 20):
    with pytest.raises(ValueError, match='{} {}: {}'.format('record' if kind == 'record' else 'compressed offset', where, ERROR_CASES[case])):
      process_bam(bam, str(d / 'out'), threads=3, chunk_bytes=chunk)
    assert os.listdir(str(d)) == ['bad.bam']


def test_options_out_of_range(engine, edge_bams):  # noqa: F811
  for kw in ({'max_d': -1}, {'max_d': 10001}, {'max_size': 10001}):
    with pytest.raises(RuntimeError):
      engine.alignment_error_counts(edge_bams['perfect'], **kw)


# ---- round trip and command line ---------------------------------------------------------------------------------

def test_round_trip_counts_every_variant_entry(config5_bams):  # noqa: F811
  """generate-reads --corrupt -> god-aligner (the config5 fixture) -> alignment-analysis: the v_size row totals are
  the v_list entries of the FASTQ pair's qnames (parse_qname), each read with its own fields, binned by size."""
  from mitty_b200.benchmarking.alignment_analysis import process_bam
  from mitty_b200.simulation.readgenerate import parse_qname
  bam = config5_bams['normal', True]
  d = os.path.dirname(bam)
  res = process_bam(bam, max_size=10, threads=4)
  want = np.zeros(24, dtype=np.uint64)
  n = 0
  for f, fq in enumerate(('normal.1.fq', 'normal.2.fq')):
    with open(os.path.join(d, fq)) as fp:
      for i, line in enumerate(fp):
        if i % 4:
          continue
        vl = parse_qname(line[1:].rstrip('\n'))[f].v_list
        n += 1
        for v in vl:
          want[min(max(v, -11), 11) + 11] += 1
        if not vl:
          want[23] += 1
  assert res['records'] == n and res['exact'] == n
  assert np.array_equal(res['vsize'].sum(axis=1), want) and want[:23].sum() > 100


def test_cli_file_and_fifo(tmp_path, edge_bams):  # noqa: F811
  from click.testing import CliRunner
  from mitty_b200.benchmarking.alignment_analysis import read_csv
  from mitty_b200.cli import cli
  bam = edge_bams['corrupt']
  want = A.analysis(open(bam, 'rb').read(), max_d=7, max_size=4)
  prefix = str(tmp_path / 'f')
  res = CliRunner().invoke(cli, ['alignment-analysis', bam, prefix, '--max-d', '7', '--max-size', '4', '--threads', '3'], catch_exceptions=False)
  assert res.exit_code == 0 and 'records analysed' in res.output, res.output
  for suffix, key in (('.mq.csv', 'mq'), ('.vsize.csv', 'vsize')):
    assert np.array_equal(read_csv(prefix + suffix)[2], want[key])
  fifo = str(tmp_path / 'in.bam')
  os.mkfifo(fifo)

  def feed():
    with open(fifo, 'wb') as fp:
      fp.write(open(bam, 'rb').read())

  th = threading.Thread(target=feed)
  th.start()
  prefix2 = str(tmp_path / 'p')
  res = CliRunner().invoke(cli, ['alignment-analysis', fifo, prefix2, '--max-d', '7', '--max-size', '4', '--threads', '3'], catch_exceptions=False)
  th.join()
  assert res.exit_code == 0, res.output
  for suffix in ('.mq.csv', '.vsize.csv'):
    assert open(prefix + suffix).read() == open(prefix2 + suffix).read()
