"""bam2illumina on the device: every count equals the pure-Python specification (tests/read_model_spec.py) on
god-aligner BAMs and hand-built BAMs, whatever the BGZF layout, chunk size and inflate threads; malformed
input raises ValueError naming the record or offset and leaves nothing behind; a model built from the BAM of
reads simulated with a shipped model reproduces that model within the DKW bound and drives generate-reads."""
import math
import os
import struct
import threading
import time

import numpy as np
import pytest

from mitty_b200 import synth
from tests import helpers as H
from tests import read_model_spec as S
from tests.test_read_model_spec import _raw, _rules_records

pytestmark = pytest.mark.gpu

GOLDEN = {'perfect': ('edge.r1.fq.gz', 'edge.r2.fq.gz'), 'corrupt': ('edge.c1.fq.gz', 'edge.c2.fq.gz')}
COUNTERS = ('records', 'considered', 'counted') + S.SKIPS


@pytest.fixture(scope='module')
def engine():
  from mitty_b200.engine import Engine
  e = Engine(0)
  yield e
  e.close()


def _same(got, want):
  for k in ('bq_mat', 'len_hist', 'tlen'):
    assert got[k].dtype == np.uint64 and np.array_equal(got[k], want[k]), k
  assert {k: got[k] for k in COUNTERS} == {k: want[k] for k in COUNTERS}


def _check(engine, path, **kw):
  data = open(path, 'rb').read()
  got = engine.read_model_counts(path, **kw)
  spec_kw = {k: v for k, v in kw.items() if k in ('max_bp', 'max_tlen', 'min_mq', 'every')}
  _same(got, S.counts(data, **spec_kw))
  assert got['inflated_bytes'] == sum(len(r) for _, r in S.members(data)) and got['compressed_bytes'] == len(data)
  return got


def _god_aligner(fasta, bam, fq1, fq2=None):
  import mitty_b200.benchmarking.god_aligner as ga
  ga.process_multi_threaded(fasta, bam, fq1, fq2, threads=4, level=1)
  return bam


@pytest.fixture(scope='module')
def edge_bams(tmp_path_factory):
  d = tmp_path_factory.mktemp('edge')
  fa, _, _ = synth.write_workload(synth.edge_workload(), str(d / 'edge'))
  return {kind: _god_aligner(fa, str(d / (kind + '.bam')), *(os.path.join(H.GOLDEN, n) for n in GOLDEN[kind])) for kind in GOLDEN}


@pytest.mark.parametrize('kind', sorted(GOLDEN))
@pytest.mark.parametrize('every', [1, 3, 7])
@pytest.mark.parametrize('min_mq', [0, 30])
def test_golden_edge_bams(engine, edge_bams, kind, every, min_mq):
  got = _check(engine, edge_bams[kind], every=every, min_mq=min_mq, threads=4)
  assert got['counted'] > 0 and got['eof_marker'] == 1


@pytest.fixture(scope='module')
def config5_bams(tmp_path_factory):
  import mitty_b200.simulation.illumina as il
  import mitty_b200.simulation.readgenerate as rg
  d = tmp_path_factory.mktemp('config5')
  mix = synth.config5()
  m = H.model('hiseq-X-v2.5-Garvan.pkl')
  out = {}
  for name, seed in (('normal', 7), ('tumor', 8)):
    wl = mix[name]
    fa, vcf, bed = synth.write_workload(wl, str(d / name))
    r1, r2, s1 = (str(d / (name + x)) for x in ('.1.fq', '.2.fq', '.s.fq'))
    rg.process_multi_threaded(fa, vcf, wl['sample'], bed, il, m, 8.0, r1, r2, threads=1, seed=seed, mode='philox', corrupt=True)
    rg.process_multi_threaded(fa, vcf, wl['sample'], bed, il, m, 8.0, s1, None, threads=1, seed=seed + 10, mode='philox', corrupt=True)
    out[name, True] = _god_aligner(fa, str(d / (name + '.p.bam')), r1, r2)
    out[name, False] = _god_aligner(fa, str(d / (name + '.s.bam')), s1)
  return out


@pytest.mark.parametrize('name', ['normal', 'tumor'])
@pytest.mark.parametrize('paired', [True, False])
def test_config5(engine, config5_bams, name, paired):
  got = _check(engine, config5_bams[name, paired], threads=8)
  assert got['counted'] == got['records']
  assert (got['tlen'].sum() > 0) == paired


def _hand_built():
  """Every skip reason, both mates, reverse strand, q > 93, |TLEN| >= max_tlen, negative and INT32_MIN TLEN,
  reads longer than max_bp, among random records."""
  raw, _ = _raw(3000, seed=5)
  rng = np.random.RandomState(6)
  extra = _rules_records() + [S.record(flag=int(f), seq=b'A' * int(l), qual=[int(q) for q in rng.randint(0, 256, int(l))], tlen=int(t),
                                       mapq=int(rng.randint(0, 61)))
                              for f, l, t in zip(rng.choice([0x41, 0x51, 0x81, 0x91, 0x61, 0xA1], 500), rng.randint(1, 400, 500),
                                                 rng.choice([-2 ** 31, 2 ** 31 - 1, -999, 999, 1000, -1000, 0, 5], 500))]
  return raw + b''.join(extra)


@pytest.mark.parametrize('every', [1, 3, 7])
@pytest.mark.parametrize('min_mq', [0, 30])
def test_hand_built(engine, tmp_path, every, min_mq):
  p = str(tmp_path / 'h.bam')
  open(p, 'wb').write(S.bgzf(_hand_built(), cuts=9000))
  got = _check(engine, p, every=every, min_mq=min_mq, threads=3)
  if every == 1 and min_mq == 30:                                  # the inputs reach every rule
    assert all(got[k] > 0 for k in S.SKIPS) and got['bq_mat'][:, :, 93].sum() > 0 and got['bq_mat'][1].sum() > 0
  wide = _check(engine, p, every=every, min_mq=min_mq, max_bp=700, max_tlen=50, threads=3)   # stripes of cycles when max_bp > 300
  assert wide['skip_long'] == 0


LAYOUTS = {
  'fixed': dict(cuts=65280),
  'random': None,
  'one_byte_and_empty': dict(cuts=[1, 1, 1, 37, 1, 4096, 1, 2] * 3, empty_every=2),
  'level0': dict(cuts=30000, level=0),
  'extra_subfields': dict(cuts=20000, extra=b'XY\x03\x00abc'),
}


@pytest.mark.parametrize('layout', sorted(LAYOUTS))
def test_layout_chunks_threads_do_not_matter(engine, tmp_path, layout):
  raw = _hand_built()
  if LAYOUTS[layout] is None:
    rng = np.random.RandomState(8)
    cuts = np.cumsum(rng.randint(0, 30000, 200))
    cuts = np.diff(np.concatenate([[0], cuts[cuts < len(raw)]]))
    data = S.bgzf(raw, cuts=[int(x) for x in cuts], level=lambda k: int(rng.randint(0, 10)), empty_every=7)
  else:
    data = S.bgzf(raw, **LAYOUTS[layout])
  p = str(tmp_path / 'l.bam')
  open(p, 'wb').write(data)
  want = S.counts(data)
  for threads in (1, 3, 16):
    for chunk in (1 << 17, 1 << 20, 64 << 20):
      got = engine.read_model_counts(p, threads=threads, chunk_bytes=chunk)
      _same(got, want)
      if chunk == 1 << 17:
        assert got['chunks'] >= len(raw) // (1 << 17)


def _device_tampered(case):
  raw = _hand_built()
  recs = S.records(raw)
  start = len(raw) - sum(len(r) for r in recs)
  k = next(i for i in range(1000, len(recs)) if len(recs[i]) < 250 and struct.unpack_from('<i', recs[i], 20)[0] > 3)
  at = start + sum(len(r) for r in recs[:k])
  r = bytearray(recs[k])
  bs, l_name, n_cig = struct.unpack_from('<i', r, 0)[0], r[12], struct.unpack_from('<H', r, 16)[0]
  rem = bs - 32 - l_name - 4 * n_cig
  if case == 'name':
    r[12] = 255
  elif case == 'cigar':
    struct.pack_into('<H', r, 16, 0xFFFF)
  elif case == 'seq':
    struct.pack_into('<i', r, 20, 2 * rem + 1)
  elif case == 'qual':
    struct.pack_into('<i', r, 20, rem)
  elif case == 'l_seq_int32_max':                   # (l_seq + 1) / 2 must not wrap in 32 bits
    struct.pack_into('<i', r, 20, 2 ** 31 - 1)
  else:
    struct.pack_into('<i', r, 20, -5)
  return raw[:at] + bytes(r) + raw[at + len(r):], k


DEVICE_CASES = {'name': 'read name', 'cigar': 'CIGAR', 'seq': 'SEQ', 'qual': 'QUAL', 'negative_l_seq': 'SEQ', 'l_seq_int32_max': 'SEQ'}


@pytest.mark.parametrize('case', sorted(DEVICE_CASES) + ['not_gzip', 'crc', 'isize', 'truncated_member', 'magic', 'block_size', 'cut_record'])
def test_errors_name_the_record_or_offset(tmp_path, case):
  from mitty_b200.empirical.bam2illumina import process_bam_parallel
  from tests.test_read_model_spec import _tampered
  if case in DEVICE_CASES:
    raw, k = _device_tampered(case)
    data, (kind, where) = S.bgzf(raw, cuts=7000), ('record', k)
  else:
    data, (kind, where) = _tampered(case)
  with pytest.raises(S.SpecError) as e:
    S.counts(data)
  assert (e.value.kind, e.value.where) == (kind, where)
  if case in DEVICE_CASES:
    assert str(e.value).endswith(DEVICE_CASES[case] + ' overruns')
  d = tmp_path / 'e'
  d.mkdir()
  bam, pkl = str(d / 'bad.bam'), str(d / 'bad.pkl')
  open(bam, 'wb').write(data)
  for chunk in (1 << 17, 64 << 20):
    with pytest.raises(ValueError, match='{} {}:'.format('record' if kind == 'record' else 'compressed offset', where)) as e:
      process_bam_parallel(bam, pkl, 'bad', threads=3, chunk_bytes=chunk)
    if case in DEVICE_CASES:
      assert str(e.value).endswith(DEVICE_CASES[case] + ' overruns block_size')
    assert os.listdir(str(d)) == ['bad.bam']                 # no .pkl, no temporary file


def test_a_malformed_record_stops_the_reading(tmp_path):
  """A record the device rejects ends the input: the rest of a FIFO that would only arrive later is not
  waited for (the writer holds it back for a minute), and the error names the record."""
  from mitty_b200.empirical.bam2illumina import process_bam_parallel
  good = S.record(name=b'r', flag=0x41, seq=b'ACGT' * 40, qual=[30] * 160, tlen=300)
  bad = bytearray(good)
  bad[12] = 255                                      # read name overruns block_size
  data = S.bgzf(S.header() + good * 5 + bytes(bad) + good * 12000, cuts=65280, level=0)
  head, tail = data[:2 << 20], data[2 << 20:]        # many 128 KiB chunks before the pause
  fifo, pkl = str(tmp_path / 'in.bam'), str(tmp_path / 'out.pkl')
  os.mkfifo(fifo)
  release = threading.Event()

  def feed():
    try:
      with open(fifo, 'wb') as fp:
        fp.write(head)
        fp.flush()
        release.wait(60)
        fp.write(tail)
    except BrokenPipeError:                          # the reader stopped and closed its end
      pass

  th = threading.Thread(target=feed)
  th.start()
  t0 = time.time()
  try:
    with pytest.raises(ValueError, match='record 5: read name overruns block_size'):
      process_bam_parallel(fifo, pkl, 'bad', threads=2, chunk_bytes=1 << 17)
    assert time.time() - t0 < 30
  finally:
    release.set()
    th.join()
  assert os.listdir(str(tmp_path)) == ['in.bam']


def test_nothing_counted_writes_nothing(tmp_path):
  from mitty_b200.empirical.bam2illumina import process_bam_parallel
  bam, pkl = str(tmp_path / 'u.bam'), str(tmp_path / 'u.pkl')
  open(bam, 'wb').write(S.bgzf(S.header() + S.record(flag=4) * 3))
  with pytest.raises(ValueError, match='no read was counted'):
    process_bam_parallel(bam, pkl, 'none')
  assert os.listdir(str(tmp_path)) == ['u.bam']


def _dkw(n, alpha):
  return math.sqrt(math.log(2 / alpha) / (2 * n))


def test_round_trip_reproduces_the_model(tmp_path):
  """Garvan -> generate-reads on an N-free, variant-free 3 Mb contig -> corrupt-reads (file k uses cum_bq_mat[k])
  -> god-aligner -> bam2illumina: every (mate, cycle) row and the template lengths >= the read length follow the
  model within the DKW bound (alpha = 1e-9 over all rows) plus the 16-bit quantisation of the alias tables."""
  import mitty_b200.simulation.illumina as il
  import mitty_b200.simulation.readcheck as chk
  import mitty_b200.simulation.readcorrupt as rc
  import mitty_b200.simulation.readgenerate as rg
  from click.testing import CliRunner
  from mitty_b200.cli import cli
  from mitty_b200.readmodels import get_read_model, load_model
  L = 3000000
  wl = {'contigs': [('rt', synth.synth_contig(L, 5))], 'tables': [synth._empty_table('rt', 2)], 'regions': [('rt', 0, L)], 'sample': 'RT'}
  fa, vcf, bed = synth.write_workload(wl, str(tmp_path / 'rt'))
  raw_model = load_model('hiseq-X-v2.5-Garvan.pkl')
  r1, r2, c1, c2 = (str(tmp_path / n) for n in ('r1.fq', 'r2.fq', 'c1.fq', 'c2.fq'))
  rg.process_multi_threaded(fa, vcf, 'RT', bed, il, raw_model, 5.0, r1, r2, threads=1, seed=3, mode='philox')
  rc.multi_process(il, raw_model, r1, c1, r2, c2, seed=4)
  bam = _god_aligner(fa, str(tmp_path / 'rt.bam'), c1, c2)
  pkl = str(tmp_path / 'rt.pkl')
  res = CliRunner().invoke(cli, ['create-read-model', 'bam2illumina', bam, pkl, 'round trip', '--threads', '4'], catch_exceptions=False)
  assert res.exit_code == 0 and 'records counted' in res.output, res.output
  m = load_model(pkl)
  assert (m['min_rlen'], m['max_rlen'], m['mean_rlen']) == (150, 150, 150)
  bq = m['bq_mat']
  assert not bq[:, 150:].any() and not m['cum_bq_mat'][:, 150:].any()
  alpha, slack = 1e-9 / (2 * 150 + 1), 2.0 ** -14
  for mate in (0, 1):
    for c in range(150):
      n = int(bq[mate, c].sum())
      assert n > 20000
      emp = np.cumsum(bq[mate, c]) / n
      assert np.abs(emp - raw_model['cum_bq_mat'][mate, c]).max() <= _dkw(n, alpha) + slack, (mate, c)
  # template lengths: tl = searchsorted(cum_tlen, u) = te - ts, which is |TLEN| of a variant-free haplotype when tl >= rlen
  t = m['tlen'][150:].astype(np.float64)
  ct = raw_model['cum_tlen']
  want = (ct[150:] - ct[149]) / (1 - ct[149])
  assert np.abs(np.cumsum(t) / t.sum() - want).max() <= _dkw(t.sum(), alpha) + slack
  # the new model drives generate-reads, and the reads re-derive from their qnames
  module, model = get_read_model(pkl)
  g1, g2 = str(tmp_path / 'g1.fq'), str(tmp_path / 'g2.fq')
  rg.process_multi_threaded(fa, vcf, 'RT', bed, module, model, 1.0, g1, g2, threads=1, seed=9, mode='philox')
  chk_res = chk.check_fastq(fa, vcf, 'RT', bed, g1, g2)
  assert chk_res['bad'] == 0 and chk_res['reads'] > 0


def test_cli_file_and_fifo(tmp_path, edge_bams):
  from click.testing import CliRunner
  from mitty_b200.cli import cli
  from mitty_b200.readmodels import load_model
  bam = edge_bams['corrupt']
  pkl = str(tmp_path / 'f.pkl')
  res = CliRunner().invoke(cli, ['create-read-model', 'bam2illumina', bam, pkl, 'edge', '--threads', '3', '--every', '3', '--min-mq', '30'],
                           catch_exceptions=False)
  assert res.exit_code == 0 and 'records counted' in res.output, res.output
  want = S.counts(open(bam, 'rb').read(), every=3, min_mq=30)
  m = load_model(pkl)
  assert np.array_equal(m['bq_mat'], want['bq_mat']) and np.array_equal(m['tlen'], want['tlen']) and m['min_mq'] == 30
  fifo = str(tmp_path / 'in.bam')
  os.mkfifo(fifo)

  def feed():
    with open(fifo, 'wb') as fp:
      fp.write(open(bam, 'rb').read())

  th = threading.Thread(target=feed)
  th.start()
  pkl2 = str(tmp_path / 'p.pkl')
  res = CliRunner().invoke(cli, ['create-read-model', 'bam2illumina', fifo, pkl2, 'edge', '--threads', '3', '--every', '3', '--min-mq', '30'],
                           catch_exceptions=False)
  th.join()
  assert res.exit_code == 0, res.output
  m2 = load_model(pkl2)
  assert all(np.array_equal(m[k], m2[k]) if isinstance(m[k], np.ndarray) else m[k] == m2[k] for k in m)
