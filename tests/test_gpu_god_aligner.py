"""god-aligner on the device: the BAM and BAI equal the pure-Python specification (tests/bam_spec.py) byte
for byte on the reference's golden FASTQ and on generated config5 workloads, and do not depend on the run
size, the chunk size or the deflate threads."""
import glob
import gzip
import os
import threading

import pytest

from mitty_b200 import synth
from tests import bam_spec as S
from tests import helpers as H

pytestmark = pytest.mark.gpu

GOLDEN = {'perfect': ('edge.r1.fq.gz', 'edge.r2.fq.gz'), 'corrupt': ('edge.c1.fq.gz', 'edge.c2.fq.gz')}


def _contigs(wl):
  return [(n, int(s.shape[0])) for n, s in wl['contigs']]


@pytest.fixture(scope='module')
def edge(tmp_path_factory):
  d = tmp_path_factory.mktemp('edge')
  wl = synth.edge_workload()
  fa, vcf, bed = synth.write_workload(wl, str(d / 'edge'))
  return {'wl': wl, 'fasta': fa, 'vcf': vcf, 'bed': bed, 'contigs': _contigs(wl)}


def _run(fasta, bam, fq1, fq2=None, **kw):
  import mitty_b200.benchmarking.god_aligner as ga
  return ga.process_multi_threaded(fasta, bam, fq1, fq2, **kw)


def _check(bam, contigs, fq1, fq2=None):
  data = open(bam, 'rb').read()
  assert S.decompress(data) == S.bam_bytes(contigs, fq1, fq2)
  assert open(bam + '.bai', 'rb').read() == S.build_bai(data, len(contigs))
  return data


@pytest.mark.parametrize('kind', ['perfect', 'corrupt'])
def test_golden_edge(tmp_path, edge, kind):
  f1, f2 = (os.path.join(H.GOLDEN, n) for n in GOLDEN[kind])
  bam = str(tmp_path / 'g.bam')
  res = _run(edge['fasta'], bam, f1, f2, threads=4)
  assert res['records'] == 2 * H.golden_fastq(GOLDEN[kind][0]).count(b'\n') // 4
  _check(bam, edge['contigs'], H.golden_fastq(GOLDEN[kind][0]), H.golden_fastq(GOLDEN[kind][1]))


@pytest.fixture(scope='module')
def config5(tmp_path_factory):
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
    rg.process_multi_threaded(fa, vcf, wl['sample'], bed, il, m, 8.0, r1, r2, threads=1, seed=seed, mode='philox')
    rg.process_multi_threaded(fa, vcf, wl['sample'], bed, il, m, 8.0, s1, None, threads=1, seed=seed + 10, mode='philox', corrupt=True)
    out[name] = {'fasta': fa, 'contigs': _contigs(wl), 'r1': r1, 'r2': r2, 's1': s1}
  return out


@pytest.mark.parametrize('name', ['normal', 'tumor'])
@pytest.mark.parametrize('paired', [True, False])
def test_config5(tmp_path, config5, name, paired):
  w = config5[name]
  bam = str(tmp_path / 'c.bam')
  f1, f2 = (w['r1'], w['r2']) if paired else (w['s1'], None)
  _run(w['fasta'], bam, f1, f2)
  _check(bam, w['contigs'], open(f1, 'rb').read(), open(f2, 'rb').read() if f2 else None)


def test_output_does_not_depend_on_runs_chunks_threads(tmp_path, config5):
  w = config5['normal']
  one = str(tmp_path / 'one.bam')
  res = _run(w['fasta'], one, w['r1'], w['r2'], threads=8)
  assert res['runs'] == 1
  ref = (open(one, 'rb').read(), open(one + '.bai', 'rb').read())
  d = tmp_path / 'many'
  d.mkdir()
  for run_bytes, chunk, threads in ((3 << 19, 1 << 20, 1), (2 << 20, 333333, 5)):
    bam = str(d / 'm.bam')
    res = _run(w['fasta'], bam, w['r1'], w['r2'], threads=threads, run_bytes=run_bytes, chunk_bytes=chunk)
    assert res['runs'] >= 4, res
    assert (open(bam, 'rb').read(), open(bam + '.bai', 'rb').read()) == ref
    assert sorted(os.listdir(str(d))) == ['m.bam', 'm.bam.bai']        # no temporary run file remains


def test_round_trip_to_fastq(tmp_path, edge):
  import mitty_b200.simulation.readcheck as chk
  f1, f2 = (os.path.join(H.GOLDEN, n) for n in GOLDEN['perfect'])
  bam = str(tmp_path / 'r.bam')
  _run(edge['fasta'], bam, f1, f2, run_bytes=1 << 20)
  reads = S.decode_reads(S.decompress(open(bam, 'rb').read()))
  got = {(name, flag & 0xC0): (seq, qual) for name, flag, seq, qual in reads}
  iupac = set(b'=ACMGRSVTWYHKDBN')
  for which, fn in enumerate(GOLDEN['perfect']):
    for name, seq, qual in S.fastq_records(H.golden_fastq(fn)):
      want = bytes(c if c in iupac else ord('N') for c in seq.upper())
      assert got.pop((name, 0x40 << which)) == (want, qual)
  assert not got
  res = chk.check_fastq(edge['fasta'], edge['vcf'], edge['wl']['sample'], edge['bed'], f1, f2)
  assert res['bad'] == 0 and res['reads'] == len(reads)


def _tamper(buf, rec, fn):
  lines = buf.split(b'\n')
  lines[4 * rec] = fn(lines[4 * rec])
  return b'\n'.join(lines)


@pytest.mark.parametrize('case', ['chrom', 'long_name', 'cigar', 'past_end'])
def test_errors_name_the_record(tmp_path, edge, case):
  lengths = dict(edge['contigs'])

  def fn(q):
    f = q.split(b'|')
    if case == 'chrom':
      f[1] = b'nosuchcontig'
    elif case == 'long_name':
      f[-1] += b',0' * 130
    elif case == 'cigar':
      f[6] = f[6][:-1] + b'Q'
    else:
      f[4] = str(lengths[f[1].decode()] - 20).encode()
    return b'|'.join(f)

  d = tmp_path / 'e'
  d.mkdir()
  fq = str(d / 'bad.fq')
  open(fq, 'wb').write(_tamper(H.golden_fastq('edge.r1.fq.gz'), 5000, fn))
  bam = str(d / 'bad.bam')
  with pytest.raises(ValueError, match='record 5001') as e:
    _run(edge['fasta'], bam, fq, run_bytes=1 << 20, chunk_bytes=1 << 18)
  assert '@EDGE:0:16:88|' in str(e.value)
  assert sorted(os.listdir(str(d))) == ['bad.fq']                         # no BAM, no index, no temporary file


def test_cli_gzip_and_fifo_inputs(tmp_path, edge):
  from click.testing import CliRunner
  from mitty_b200.cli import cli
  f1, f2 = (os.path.join(H.GOLDEN, n) for n in GOLDEN['corrupt'])
  bam = str(tmp_path / 'cli.bam')
  res = CliRunner().invoke(cli, ['god-aligner', edge['fasta'], f1, bam, '--fastq2', f2, '--threads', '3', '--level', '1'], catch_exceptions=False)
  assert res.exit_code == 0 and 'records written' in res.output, res.output
  ref = _check(bam, edge['contigs'], H.golden_fastq(GOLDEN['corrupt'][0]), H.golden_fastq(GOLDEN['corrupt'][1]))
  p1, p2 = str(tmp_path / 'p1'), str(tmp_path / 'p2')
  os.mkfifo(p1); os.mkfifo(p2)

  def feed(path, data):
    with open(path, 'wb') as fp:
      fp.write(data)

  th = [threading.Thread(target=feed, args=(p, gzip.compress(H.golden_fastq(n)) if k == 0 else H.golden_fastq(n)))
        for k, (p, n) in enumerate(zip((p1, p2), GOLDEN['corrupt']))]
  for t in th:
    t.start()
  fbam = str(tmp_path / 'fifo.bam')
  res = CliRunner().invoke(cli, ['god-aligner', edge['fasta'], p1, fbam, '--fastq2', p2, '--threads', '3', '--level', '1'], catch_exceptions=False)
  for t in th:
    t.join()
  assert res.exit_code == 0, res.output
  assert open(fbam, 'rb').read() == ref and open(fbam + '.bai', 'rb').read() == open(bam + '.bai', 'rb').read()
  assert not glob.glob(str(tmp_path / '*.run*'))
