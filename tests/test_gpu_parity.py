"""GPU parity tests (run on the B200 box with -m gpu).  Everything goes through the C ABI
(libmitty_b200.so) and is compared with the oracle / the golden vectors of the reference:
bit-exact for every byte and index."""
import os

import numpy as np
import pytest

import oracle
from mitty_b200 import synth
from mitty_b200.lib import vcfio
from tests import helpers as H
from tests.test_oracle_golden import RPC_KAT_CPY0, RPC_KAT_CPY1

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def eng():
  from mitty_b200.engine import Engine
  e = Engine(0)
  yield e
  e.close()


def gpu_generate(eng, wl, model, coverage, seed, mode, corrupt=False, regions=None):
  """In-memory generate-reads: the loop of readgenerate.process_multi_threaded without files."""
  import mitty_b200.simulation.illumina as il
  import mitty_b200.simulation.readgenerate as rg
  regions = regions or H.workload_regions(wl)
  rm = il.read_model_params(model, coverage)
  eng.load_model(rm)
  cache = rg.RegionCache(eng, regions, None)
  cache.fetch_ref = lambda region: next(r['ref'] for r in regions if r['region'] == region)
  o1, o2, total = [], [], 0
  for ps, wd in enumerate(rg.get_data_for_workers(rm, regions, seed)):
    r_idx, cpy = wd['region_idx'], wd['region_cpy']
    cp = cache.copy(r_idx, cpy)
    f1, f2, cnt, _, _ = rg.generate_unit(eng, il, rm, cp, regions[r_idx]['region'][0], cpy, int(wd['rng_seed']), wl['sample'], 0, ps,
                                         mode=mode, corrupt=corrupt, corrupt_seed=seed)
    o1.append(f1.tobytes()); o2.append(f2.tobytes()); total += cnt
  for cp in cache.copies.values():
    eng.free_copy(cp)
  for rid in cache.regions.values():
    eng.free_region(rid)
  return b''.join(o1), b''.join(o2), total


# ---- the reference's own KATs through the device ---------------------------------------------------

def test_tiny_node_list_and_reads(eng, tmp_path):
  """test_rpc.py:111-180 through mg_copy_build / k_hap_build / k_unit_emit."""
  import mitty_b200.simulation.rpc as rpc
  p = H.write_tiny(tmp_path)
  vcf = vcfio.load_variant_file(p['vcf'], 'g0_s0', p['whole_bed'])
  nl = rpc.create_node_list(H.TINY_SEQ, 1, vcf[0]['v'][1], engine=eng)
  assert nl.tuples() == [
    (1, 1, '=', 4, 'ATGA', None), (5, 5, 'X', 1, 'T', 0), (6, 6, '=', 3, 'GTA', None),
    (9, 9, 'I', 3, 'TTT', 3), (12, 9, '=', 3, 'TCC', None), (14, 14, 'D', 2, '', -2),
    (15, 14, '=', 7, 'GGAGGCG', None), (21, 25, 'D', 4, '', -4), (22, 25, '=', 1, 'C', None)]
  for pp, l, n0, n1, want in RPC_KAT_CPY1:
    got = rpc.generate_read(pp, l, nl)
    if got is not None:   # None: template end on/after p_max, never sampled by the reference
      assert got == want
  assert rpc.generate_read(9, 2, nl) == (8, '>0:2I', [3], 'TT')
  assert rpc.generate_read(1, 10, nl) == (1, '4=1X3=2I', [0, 3], 'ATGATGTATT')
  nl.free()
  nl = rpc.create_node_list(H.TINY_SEQ, 1, vcf[0]['v'][0], engine=eng)
  for pp, l, n0, n1, want in RPC_KAT_CPY0:
    assert rpc.generate_read(pp, l, nl) == want
  nl.free()


def test_edge_nodes_and_haplotypes(eng):
  """Node tables and packed haplotypes of every (region, copy) of the edge workload == oracle."""
  import mitty_b200.simulation.rpc as rpc
  for r in H.workload_regions(synth.edge_workload()):
    for vl in r['v']:
      nl = rpc.create_node_list(r['ref'], r['region'][1] + 1, vl, engine=eng)
      assert nl.tuples() == oracle.create_node_list(r['ref'], r['region'][1] + 1, H.oracle_cv(vl))
      nl.free()


@pytest.mark.parametrize('seed', [1, 2, 3, 4])
def test_device_walk_dense_overlapping_variants(eng, seed):
  """The device node-list walk (chain marking by pointer doubling) against the oracle's sequential
  walk on variant sets built to stress the greedy skip rule (rpc.py:55): long deletions that swallow
  runs of later variants, chains of overlapping deletions, several records at one POS, variants
  before the region start, non-ACGT bytes in ALT alleles and in the reference."""
  import mitty_b200.simulation.rpc as rpc
  region, bed_start, vl, n_recs = H.dense_variant_region(seed)
  want = oracle.create_node_list(region, bed_start + 1, H.oracle_cv(vl))
  assert want[-1][2] == '=' and sum(1 for w in want if w[2] != '=') < n_recs     # some records were skipped
  nl = rpc.create_node_list(region, bed_start + 1, vl, engine=eng)
  assert nl.tuples() == want
  # the materialised haplotype (with its non-ACGT exception runs) is the concatenation of the node sequences
  cp = eng.build_copy(eng.load_region(region, bed_start), vl)
  assert eng.copy_haplotype(cp).tobytes().decode() == ''.join(w[4] for w in want)
  nl.free()


def test_unsorted_variants_are_rejected(eng):
  import mitty_b200.simulation.rpc as rpc
  vl = vcfio.VariantList.from_variants([vcfio.Variant(12, 'A', 'C', 'X', 0), vcfio.Variant(5, 'A', 'T', 'X', 0)])
  with pytest.raises(ValueError):
    rpc.create_node_list(H.TINY_SEQ, 1, vl, engine=eng)


def test_deletion_across_region_end_is_rejected(eng):
  import mitty_b200.simulation.rpc as rpc
  vl = vcfio.VariantList.from_variants([vcfio.Variant(20, 'GTTAC', 'G', 'D', 4)])
  with pytest.raises(ValueError):
    rpc.create_node_list(H.TINY_SEQ[:23], 1, vl, engine=eng)


# ---- template sampling (plugin generate_reads) -----------------------------------------------------

def test_generate_reads_plugin_golden(eng):
  """illumina.generate_reads (deterministic draws, device searchsorted/filter) == the reference."""
  import mitty_b200.simulation.illumina as il
  z = np.load(os.path.join(H.GOLDEN, 'templates.npz'))
  for key in sorted({k.rsplit('_', 1)[0] for k in z.files}):
    name, p_min, p_max, seed = key.rsplit('_', 3)
    rm = il.read_model_params(H.model(name + '.pkl'), 30.0)
    r = il.generate_reads(rm, int(p_min), int(p_max), int(seed), engine=eng)
    np.testing.assert_array_equal(r[0]['pos'], z[key + '_pos0'])
    np.testing.assert_array_equal(r[1]['pos'], z[key + '_pos1'])
    np.testing.assert_array_equal(r[0]['file_order'], z[key + '_fo0'])
    np.testing.assert_array_equal(r[1]['file_order'], z[key + '_fo1'])
    assert r[0]['len'].dtype == np.uint32 and (r[0]['len'] == rm['rlen']).all()
  with pytest.raises(ValueError):
    il.generate_reads(il.read_model_params(H.model('1kg-pcr-free.pkl'), 30.0), 1, 1000, 1 << 32, engine=eng)


# ---- explicit templates: every corner of the emit kernel -------------------------------------------

@pytest.mark.parametrize('L', [150, 37, 16, 1, 250, 161, 162, 305, 306])   # 161/162, 305/306: both sides of the register-window switches
def test_edge_units_explicit(eng, L):
  from mitty_b200.engine import MODE_EXPLICIT
  regs = H.workload_regions(synth.edge_workload())
  rs = np.random.RandomState(L)
  eng.load_model({'cum_tlen': np.array([1.0]), 'cum_bq_mat': np.ones((2, 300, 94)), 'rlen': L})
  total = 0
  for ri, r in enumerate(regs):
    rid = eng.load_region(r['ref'], r['region'][1])
    for cpy, vl in enumerate(r['v']):
      cp = eng.build_copy(rid, vl)
      n = 3000
      ts = rs.randint(cp.p_min - 2, cp.p_max, size=n).astype(np.int64)
      ts[:5] = cp.p_min + np.arange(5)
      tl = rs.randint(0, 3 * L + 40, size=n).astype(np.int64)
      tl[5:10] = L
      ts[5:10] = cp.p_max - L - 1 - np.arange(5)
      fo = rs.randint(0, 2, size=n).astype(np.int8)
      f1, f2, cnt, nk, nb = eng.generate_unit(cp, n, 0.5, MODE_EXPLICIT, 0, '@EDGE:0:{}:'.format(ri), '|{}|{}'.format(r['region'][0], cpy),
                                              ts=ts, tl=tl, fo=fo)
      te = ts + np.maximum(tl, L)
      keep = (te < cp.p_max) & (ts >= cp.p_min)
      assert nk == keep.sum()
      o1, o2, ocnt = oracle.generate_unit(r['ref'], r['region'][1] + 1, H.oracle_cv(vl), L, ts[keep], te[keep], fo[:keep.sum()],
                                          'EDGE:0:{}'.format(ri), r['region'][0], cpy)
      assert cnt == ocnt
      assert f1.tobytes() == o1 and f2.tobytes() == o2
      total += cnt
      eng.free_copy(cp)
    eng.free_region(rid)
  assert total > 5000


def test_empty_and_tiny_units(eng):
  from mitty_b200.engine import MODE_EXPLICIT
  eng.load_model({'cum_tlen': np.array([1.0]), 'cum_bq_mat': np.ones((2, 300, 94)), 'rlen': 10})
  rid = eng.load_region(np.frombuffer(H.TINY_SEQ.encode(), dtype=np.uint8), 0)
  cp = eng.build_copy(rid, vcfio.VariantList.from_variants([]))
  assert (cp.p_min, cp.p_max, cp.n_nodes) == (1, 26, 1)
  f1, f2, cnt, nk, nb = eng.generate_unit(cp, 0, 0.5, MODE_EXPLICIT, 0, '@s:0:0:', '|1|0',
                                          ts=np.zeros(1, np.int64), tl=np.zeros(1, np.int64), fo=np.zeros(1, np.int8))
  assert (cnt, nk, nb, f1.size, f2.size) == (0, 0, 0, 0, 0)
  f1, f2, cnt, nk, nb = eng.generate_unit(cp, 1, 0.5, MODE_EXPLICIT, 0, '@s:0:0:', '|1|0',
                                          ts=np.array([3], np.int64), tl=np.array([12], np.int64), fo=np.ones(1, np.int8))
  assert f1.tobytes() == b'@s:0:0:1|1|0|1|5|10|10=||0|3|10|10=|\nCTTGGATACG\n+\n~~~~~~~~~~\n'
  assert f2.tobytes() == b'@s:0:0:1|1|0|1|5|10|10=||0|3|10|10=|\nGACGTATCCA\n+\n~~~~~~~~~~\n'
  eng.free_copy(cp); eng.free_region(rid)


# ---- deterministic mode: byte-exact against the reference -------------------------------------------

@pytest.mark.parametrize('name,wl_fn', [('edge', synth.edge_workload), ('edge250', synth.edge_workload),
                                        ('mid', lambda: synth.config1(contig_len=100000)),
                                        ('softmask', synth.softmask_workload),
                                        ('config1', synth.config1)])
def test_deterministic_fastq_golden(eng, name, wl_fn):
  """generate-reads (+ corrupt-reads) in deterministic mode == the unmodified reference with
  --threads 1 (golden sha256 from tests/golden/make_golden.py; edge also byte-compared)."""
  import mitty_b200.simulation.illumina as il
  from mitty_b200.engine import MODE_DET
  import mitty_b200.simulation.readcorrupt as rc
  info = H.golden()['fastq'][name]
  m = H.model(info['model'])
  wl = wl_fn()
  f1, f2, n = gpu_generate(eng, wl, m, info['coverage'], info['seed'], 'deterministic')
  assert n == info['pairs']
  if name == 'edge':
    assert f1 == H.golden_fastq('edge.r1.fq.gz') and f2 == H.golden_fastq('edge.r2.fq.gz')
  assert (len(f1), H.sha256(f1)) == (info['r1']['bytes'], info['r1']['sha256'])
  assert (len(f2), H.sha256(f2)) == (info['r2']['bytes'], info['r2']['sha256'])
  if 'c1' not in info:
    return
  a1, a2 = np.frombuffer(f1, dtype=np.uint8), np.frombuffer(f2, dtype=np.uint8)
  ws = int(np.random.RandomState(info['seed']).randint(il.SEED_MAX))
  l1, l2 = rc.seq_lengths(a1), rc.seq_lengths(a2)
  lens = np.empty(2 * l1.size, dtype=np.int64); lens[0::2] = l1; lens[1::2] = l2
  eng.load_model(m)
  c1, c2, cn = eng.corrupt_fastq(a1, a2, mode=MODE_DET, draws=il.corrupt_draws(lens.tolist(), np.random.RandomState(ws)))
  assert cn == info['pairs']
  if name == 'edge':
    assert c1.tobytes() == H.golden_fastq('edge.c1.fq.gz') and c2.tobytes() == H.golden_fastq('edge.c2.fq.gz')
  assert H.sha256(c1.tobytes()) == info['c1']['sha256'] and H.sha256(c2.tobytes()) == info['c2']['sha256']


def test_corrupt_template_plugin_golden(eng):
  import mitty_b200.simulation.illumina as il
  m = H.model('hiseq-X-v2.5-Garvan.pkl')
  for case in H.golden()['corrupt_template']:
    out = il.corrupt_template(m, tuple(case['in']), np.random.RandomState(case['seed']), engine=eng)
    assert [list(o) for o in out] == case['out']


def test_corrupt_read_longer_than_model(eng):
  m = dict(H.model('hiseq-X-v2.5-Garvan.pkl'))
  eng.load_model(m)
  s = 'A' * 301
  with pytest.raises(IndexError):
    eng.corrupt_fastq('@q\n{}\n+\n{}\n'.format(s, s).encode())


def test_cli_files_deterministic(tmp_path):
  """The command line end to end on files (FASTA / VCF.gz / BED in, two FASTQ out)."""
  from click.testing import CliRunner
  from mitty_b200.cli import cli
  info = H.golden()['fastq']['edge']
  wl = synth.edge_workload()
  fa, vcf, bed = synth.write_workload(wl, str(tmp_path / 'edge'), gz=True)
  r1, r2, c1, c2 = (str(tmp_path / x) for x in ('r1.fq', 'r2.fq', 'c1.fq', 'c2.fq'))
  res = CliRunner().invoke(cli, ['generate-reads', fa, vcf, wl['sample'], bed, info['model'], str(info['coverage']), str(info['seed']),
                                 r1, '--fastq2', r2, '--threads', '1', '--deterministic'], catch_exceptions=False)
  assert res.exit_code == 0, res.output
  assert open(r1, 'rb').read() == H.golden_fastq('edge.r1.fq.gz') and open(r2, 'rb').read() == H.golden_fastq('edge.r2.fq.gz')
  res = CliRunner().invoke(cli, ['corrupt-reads', info['model'], r1, c1, str(info['seed']), '--fastq2-in', r2, '--fastq2-out', c2,
                                 '--threads', '1', '--deterministic'], catch_exceptions=False)
  assert res.exit_code == 0, res.output
  assert open(c1, 'rb').read() == H.golden_fastq('edge.c1.fq.gz') and open(c2, 'rb').read() == H.golden_fastq('edge.c2.fq.gz')


@pytest.mark.parametrize('chunk', [1000, 65536])
def test_units_streamed_through_small_ring(tmp_path, monkeypatch, chunk):
  """A unit's bytes leave the device piece by piece through the sink's page-locked slots (drain
  thread -> writer threads): slots far smaller than a unit (even smaller than a few records) must
  give the same files."""
  import mitty_b200.simulation.illumina as il
  import mitty_b200.simulation.readgenerate as rg
  monkeypatch.setattr(rg, 'CHUNK_BYTES', chunk)
  info = H.golden()['fastq']['edge']
  wl = synth.edge_workload()
  fa, vcf, bed = synth.write_workload(wl, str(tmp_path / 'edge'))
  r1, r2 = str(tmp_path / 'r1.fq'), str(tmp_path / 'r2.fq')
  rg.process_multi_threaded(fa, vcf, wl['sample'], bed, il, H.model(info['model']), info['coverage'], r1, r2,
                            threads=2, seed=info['seed'], mode='deterministic', devices=[0, 0])
  assert open(r1, 'rb').read() == H.golden_fastq('edge.r1.fq.gz') and open(r2, 'rb').read() == H.golden_fastq('edge.r2.fq.gz')


@pytest.mark.parametrize('devices', [[0, 0], [0, 0, 0], 'all'])
def test_sharded_workers_identical_output(tmp_path, devices, monkeypatch):
  """Units dealt to several GPU workers (LPT), appended in schedule order: the bytes must not
  depend on the worker count.  [0, 0]: two workers with their own contexts on one GPU (the host
  logic of the multi-GPU path on a 1-GPU box); 'all': one worker per GPU present.  With three workers the
  regions also take the large-region route (reference bytes fetched into a worker's page-locked buffer)."""
  import mitty_b200.simulation.illumina as il
  import mitty_b200.simulation.readgenerate as rg
  from mitty_b200.engine import device_count
  if devices == [0, 0, 0]:
    monkeypatch.setattr(rg, 'PIN_REGION_BYTES', 1)
    monkeypatch.setattr(rg, 'PIN_MIN_REGIONS', 1)
  info = H.golden()['fastq']['edge']
  wl = synth.edge_workload()
  fa, vcf, bed = synth.write_workload(wl, str(tmp_path / 'edge'))
  devs = list(range(device_count())) if devices == 'all' else devices
  r1, r2 = str(tmp_path / 'r1.fq'), str(tmp_path / 'r2.fq')
  rg.process_multi_threaded(fa, vcf, wl['sample'], bed, il, H.model(info['model']), info['coverage'], r1, r2,
                            threads=len(devs), seed=info['seed'], mode='deterministic', devices=devs)
  assert open(r1, 'rb').read() == H.golden_fastq('edge.r1.fq.gz') and open(r2, 'rb').read() == H.golden_fastq('edge.r2.fq.gz')
  # production mode: same bytes for 1 worker and for several
  p1, p2 = str(tmp_path / 'p1.fq'), str(tmp_path / 'p2.fq')
  rg.process_multi_threaded(fa, vcf, wl['sample'], bed, il, H.model(info['model']), info['coverage'], p1, p2,
                            threads=len(devs), seed=5, mode='philox', corrupt=True, devices=devs)
  q1, q2 = str(tmp_path / 'q1.fq'), str(tmp_path / 'q2.fq')
  rg.process_multi_threaded(fa, vcf, wl['sample'], bed, il, H.model(info['model']), info['coverage'], q1, q2,
                            threads=1, seed=5, mode='philox', corrupt=True, devices=[0])
  assert open(p1, 'rb').read() == open(q1, 'rb').read() and open(p2, 'rb').read() == open(q2, 'rb').read()


def test_grch37_shaped_deterministic(eng):
  """BASELINE.json configs[3] at 1/500 scale: 24 GRCh37-shaped contigs with N runs, diploid
  autosomes and haploid X / Y (46 copies, 92 units): deterministic mode == the oracle's
  generate-reads + corrupt-reads, byte for byte."""
  import mitty_b200.simulation.illumina as il
  import mitty_b200.simulation.readcorrupt as rc
  from mitty_b200.engine import MODE_DET
  wl = synth.grch37_shaped(scale=0.002)
  m = H.model('hiseq-X-v2.5-Garvan.pkl')
  regs = H.workload_regions(wl)
  assert [len(r['v']) for r in regs] == [2] * 22 + [1, 1]
  f1, f2, n = gpu_generate(eng, wl, m, 30.0, 7, 'deterministic', regions=regs)
  o1, o2, on = oracle.generate_reads_cmd(H.oracle_regions(regs), m, 30.0, 7, wl['sample'])
  assert n == on and n > 400000
  assert H.sha256(f1) == H.sha256(o1) and H.sha256(f2) == H.sha256(o2)
  # corrupt a slice of it in deterministic mode (the host-side MT draws are the slow part)
  cut = f1.index(b'\n@', 20000000) + 1 if len(f1) > 20000000 else len(f1)
  nrec = f1[:cut].count(b'\n') // 4
  cut2 = len(b'\n'.join(f2.split(b'\n')[:4 * nrec])) + 1
  a1, a2 = np.frombuffer(f1[:cut], dtype=np.uint8), np.frombuffer(f2[:cut2], dtype=np.uint8)
  ws = int(np.random.RandomState(7).randint(il.SEED_MAX))
  l1, l2 = rc.seq_lengths(a1), rc.seq_lengths(a2)
  lens = np.empty(2 * l1.size, dtype=np.int64); lens[0::2] = l1; lens[1::2] = l2
  eng.load_model(m)
  c1, c2, cn = eng.corrupt_fastq(a1, a2, mode=MODE_DET, draws=il.corrupt_draws(lens.tolist(), np.random.RandomState(ws)))
  w1, w2, wn = oracle.corrupt_fastq(m['cum_bq_mat'], ws, f1[:cut], f2[:cut2])
  assert cn == wn == nrec and c1.tobytes() == w1 and c2.tobytes() == w2


@pytest.mark.parametrize('chunk', [1 << 20, 70000, 256 << 20])
def test_corrupt_reads_streaming_chunks(tmp_path, chunk):
  """corrupt-reads streams its inputs in chunks (the device reports the bytes the complete
  templates occupied, the rest is carried over): the result must not depend on the chunk size, in
  deterministic mode (== the reference golden) and in production mode (== one big chunk)."""
  import mitty_b200.simulation.illumina as il
  import mitty_b200.simulation.readcorrupt as rc
  info = H.golden()['fastq']['edge']
  m = H.model(info['model'])
  r1, r2 = str(tmp_path / 'r1.fq'), str(tmp_path / 'r2.fq.gz')
  open(r1, 'wb').write(H.golden_fastq('edge.r1.fq.gz'))
  import gzip
  with gzip.open(r2, 'wb') as fp:                       # one plain, one gzip input
    fp.write(H.golden_fastq('edge.r2.fq.gz'))
  c1, c2 = str(tmp_path / 'c1.fq'), str(tmp_path / 'c2.fq')
  rc.multi_process(il, m, r1, c1, r2, c2, processes=1, seed=info['seed'], mode='deterministic', chunk_bytes=chunk)
  assert open(c1, 'rb').read() == H.golden_fastq('edge.c1.fq.gz') and open(c2, 'rb').read() == H.golden_fastq('edge.c2.fq.gz')
  p1, p2 = str(tmp_path / 'p1.fq'), str(tmp_path / 'p2.fq')
  rc.multi_process(il, m, r1, p1, r2, p2, processes=1, seed=3, mode='philox', chunk_bytes=chunk)
  q1, q2 = str(tmp_path / 'q1.fq'), str(tmp_path / 'q2.fq')
  rc.multi_process(il, m, r1, q1, r2, q2, processes=1, seed=3, mode='philox', chunk_bytes=64 << 20)
  assert open(p1, 'rb').read() == open(q1, 'rb').read() and open(p2, 'rb').read() == open(q2, 'rb').read()
  # single-end
  s1 = str(tmp_path / 's1.fq')
  rc.multi_process(il, m, r1, s1, None, None, processes=1, seed=3, mode='philox', chunk_bytes=chunk)
  assert open(s1, 'rb').read() == open(q1, 'rb').read()


def test_tumor_normal_viral_mix(tmp_path):
  """BASELINE.json configs[4] at test scale: three generate-reads invocations (diploid normal with a
  haploid X, triploid tumour, haploid viral spike-in) concatenated the way the reference makes mixes.
  Every read must re-derive from its qname against ITS sample's haplotypes, and the per-sample pair
  counts must follow coverage x copies (each copy gets coverage / 2, illumina.py:12-40)."""
  import mitty_b200.simulation.illumina as il
  import mitty_b200.simulation.readgenerate as rg
  mix = synth.config5()
  m = H.model('hiseq-X-v2.5-Garvan.pkl')
  L = int(m['mean_rlen'])

  def expected_pairs(wl, cov):
    tables = {t.chrom: t for t in wl['tables']}
    return sum((e - s) * tables[c].gt.shape[1] * (cov / 2.0) / (2 * L) for c, s, e in wl['regions'])

  human = expected_pairs(mix['normal'], 30.0) + expected_pairs(mix['tumor'], 20.0)
  cov_v = 30.0 * (0.01 * human / 0.99) / expected_pairs(mix['virus'], 30.0)      # ~1 % of all pairs
  runs = [('normal', 30.0, 7), ('tumor', 20.0, 8), ('virus', cov_v, 9)]
  cat1, cat2 = b'', b''
  for name, cov, seed in runs:
    wl = mix[name]
    fa, vcf, bed = synth.write_workload(wl, str(tmp_path / name))
    r1, r2 = str(tmp_path / (name + '.1.fq')), str(tmp_path / (name + '.2.fq'))
    rg.process_multi_threaded(fa, vcf, wl['sample'], bed, il, m, cov, r1, r2, threads=1, seed=seed, mode='philox')
    cat1 += open(r1, 'rb').read(); cat2 += open(r2, 'rb').read()
  regs = {mix[k]['sample']: H.workload_regions(mix[k]) for k in mix}
  idx, counts, errs = {}, {}, []
  for which, buf in enumerate((cat1, cat2)):
    lines = buf.decode().split('\n')
    for k in range(0, len(lines) - 1, 4):
      info = rg.parse_qname(lines[k][1:])[which]
      key = (info.sample, info.chrom, info.cpy)
      if key not in idx:
        r = next(r for r in regs[info.sample] if r['region'][0] == info.chrom)
        idx[key] = H.HaplotypeIndex(r['ref'], r['region'][1] + 1, H.oracle_cv(r['v'][info.cpy]))
      e = idx[key].check(info, lines[k + 1])
      if e:
        errs.append((lines[k], e))
      if which == 0:
        counts[info.sample] = counts.get(info.sample, 0) + 1
  assert not errs, errs[:3]
  assert {k[0] for k in idx} == {'NORMAL', 'TUMOR', 'VIRUS'}
  assert {k[2] for k in idx if k[0] == 'TUMOR'} == {0, 1, 2} and {k[2] for k in idx if k[:2] == ('NORMAL', 'X')} == {0}
  for name, cov, _ in runs:
    exp = expected_pairs(mix[name], cov)
    got = counts[mix[name]['sample']]
    assert abs(got - exp) < 0.04 * exp + 6 * np.sqrt(exp), (name, got, exp)   # edge effects: templates need te < p_max
  frac = counts['VIRUS'] / float(sum(counts.values()))
  assert 0.006 < frac < 0.014, frac


def test_corrupt_reads_edge_inputs(eng, tmp_path):
  """corrupt-reads on the inputs the reference's reader loop meets (readcorrupt.py:49-55): empty
  files, single-end input, ragged read lengths in one file, a second file with fewer records (zip
  truncation), a last record without a trailing newline -- deterministic mode == the oracle, production
  mode == the numpy specification."""
  import mitty_b200.simulation.illumina as il
  import mitty_b200.simulation.readcorrupt as rc
  from tests import philox_ref as PR
  m = H.model('hiseq-X-v2.5-Garvan.pkl')
  eng.load_model(m)
  tables = eng.model_tables(1)
  rs = np.random.RandomState(3)

  def first_records(b, n):
    """The first n records of a FASTQ buffer, newline-terminated."""
    lines = (b if b.endswith(b'\n') else b + b'\n').split(b'\n')
    return b''.join(x + b'\n' for x in lines[:4 * n])

  def fq(lengths, tag, newline=True):
    recs = []
    for k, L in enumerate(lengths):
      seq = ''.join('ACGTNacgtR'[i] for i in rs.randint(0, 10, size=L))
      recs.append('@{}{}\n{}\n+\n{}\n'.format(tag, k, seq, '~' * L))
    s = ''.join(recs)
    return (s if newline else s[:-1]).encode()

  cases = {
    'empty': (b'', b''),
    'single': (fq([150, 150, 30, 1, 300, 75], 'a'), None),
    'ragged': (fq([150, 1, 299, 40, 150], 'b'), fq([10, 150, 150, 300, 2], 'c')),
    'shorter2': (fq([100, 100, 100, 100], 'd'), fq([100, 100], 'e')),
    'no_final_newline': (fq([50, 60], 'f', newline=False), fq([70, 80], 'g', newline=False)),
  }
  for name, (b1, b2) in cases.items():
    i1, o1 = str(tmp_path / (name + '.1.fq')), str(tmp_path / (name + '.1.out.fq'))
    open(i1, 'wb').write(b1)
    i2 = o2 = None
    if b2 is not None:
      i2, o2 = str(tmp_path / (name + '.2.fq')), str(tmp_path / (name + '.2.out.fq'))
      open(i2, 'wb').write(b2)
    rc.multi_process(il, m, i1, o1, i2, o2, processes=1, seed=11, mode='deterministic')
    want1, want2, n = oracle.corrupt_reads_cmd(m, 11, b1, b2) if b1 else (b'', b'' if b2 is not None else None, 0)
    assert open(o1, 'rb').read() == want1, name
    if b2 is not None:
      assert open(o2, 'rb').read() == want2, name
    # production mode: == the numpy specification (key 0x636f7232, read 1's name on both files), independent of the chunk size
    p1, p2 = str(tmp_path / (name + '.1.p.fq')), (str(tmp_path / (name + '.2.p.fq')) if b2 is not None else None)
    q1, q2 = str(tmp_path / (name + '.1.q.fq')), (str(tmp_path / (name + '.2.q.fq')) if b2 is not None else None)
    rc.multi_process(il, m, i1, p1, i2, p2, processes=1, seed=11)
    rc.multi_process(il, m, i1, q1, i2, q2, processes=1, seed=11, chunk_bytes=700)
    assert open(p1, 'rb').read() == open(q1, 'rb').read(), name
    r1 = first_records(b1, n)
    assert open(p1, 'rb').read() == PR.corrupt_file(r1, 0, tables, 11, 0x636f7232, names_from=r1), name
    if b2 is not None:
      assert open(p2, 'rb').read() == open(q2, 'rb').read(), name
      assert open(p2, 'rb').read() == PR.corrupt_file(first_records(b2, n), 1, tables, 11, 0x636f7232, names_from=r1), name


def test_bed_cutting_through_a_deletion(tmp_path, caplog):
  """A BED region that ends inside a deletion: the reference's node list would end in 'D' and its
  reads at the region end come out short (readgenerate.py:192).  By default that is an error raised
  before anything is written; with drop_end_deletions (--drop-end-deletions) the deletion is left out
  with a warning, every read still re-derives from its qname against the haplotype built without it,
  and regions are released after their last unit."""
  import logging
  import mitty_b200.simulation.illumina as il
  import mitty_b200.simulation.readgenerate as rg
  wl = synth.config1(contig_len=60000, names=('1',))
  seq = wl['contigs'][0][1]
  far = np.abs(wl['tables'][0].pos - 30000) > 200
  d_ref = seq[29999:30009].tobytes().decode()           # POS 30000, ten bases -> one: deletes 30001..30009
  wl['tables'][0] = synth.merge_tables(synth._subset(wl['tables'][0], far), synth.table_from_records('1', [(30000, d_ref, d_ref[0], (1, 1))], 2))
  cut = 30004                                          # 0-based end inside the deleted bases
  wl['regions'] = [('1', 1000, cut), ('1', cut + 500, 59000)]
  fa, vcf, bed = synth.write_workload(wl, str(tmp_path / 'cut'))
  r1, r2 = str(tmp_path / 'r1.fq'), str(tmp_path / 'r2.fq')
  with pytest.raises(ValueError, match='reach beyond the region end'):
    rg.process_multi_threaded(fa, vcf, wl['sample'], bed, il, H.model('hiseq-X-v2.5-Garvan.pkl'), 30.0, r1, r2, threads=1, seed=3, mode='philox')
  assert not os.path.exists(r1) and not os.path.exists(r2)          # nothing was opened, let alone truncated
  with caplog.at_level(logging.WARNING):
    rg.process_multi_threaded(fa, vcf, wl['sample'], bed, il, H.model('hiseq-X-v2.5-Garvan.pkl'), 30.0, r1, r2, threads=1, seed=3, mode='philox',
                              drop_end_deletions=True)
  assert any('reach beyond the region end' in rec.getMessage() for rec in caplog.records)
  regs = H.workload_regions(wl)
  idx = {}
  def index_for(chrom, cpy, pos):
    r = regs[0] if pos <= cut else regs[1]
    key = (r['region'], cpy)
    if key not in idx:
      idx[key] = H.HaplotypeIndex(r['ref'], r['region'][1] + 1, H.oracle_cv(rg._without_end_crossing_deletions(r['v'][cpy], r['region'], True)[0]))
    return idx[key]
  n = 0
  for which, path in enumerate((r1, r2)):
    lines = open(path).read().split('\n')
    for k in range(0, len(lines) - 1, 4):
      info = rg.parse_qname(lines[k][1:])[which]
      assert index_for(info.chrom, info.cpy, info.pos).check(info, lines[k + 1]) is None, lines[k]
      n += 1
  assert n > 5000


@pytest.mark.timeout(300)
def test_fifo_pipeline_like_the_reference_example(tmp_path):
  """examples/reads/run.sh:13-16 of the reference: generate-reads writes into two FIFOs, corrupt-reads
  reads them (`<(cat < tf1)`) and writes into two more pipes.  Everything is sequential I/O on
  streams that can be opened exactly once; the result must equal the reference's golden files."""
  import threading
  import mitty_b200.simulation.illumina as il
  import mitty_b200.simulation.readcorrupt as rc
  import mitty_b200.simulation.readgenerate as rg
  info = H.golden()['fastq']['edge']
  m = H.model(info['model'])
  wl = synth.edge_workload()
  fa, vcf, bed = synth.write_workload(wl, str(tmp_path / 'edge'))
  tf1, tf2, of1, of2 = (str(tmp_path / x) for x in ('tf1', 'tf2', 'of1', 'of2'))
  for f in (tf1, tf2, of1, of2):
    os.mkfifo(f)
  got, errs = {}, []

  def drain(name, path):
    with open(path, 'rb') as fp:
      got[name] = fp.read()

  def generate():
    try:
      rg.process_multi_threaded(fa, vcf, wl['sample'], bed, il, m, info['coverage'], tf1, tf2, threads=1, seed=info['seed'], mode='deterministic')
    except BaseException as e:  # noqa: B902
      errs.append(e)

  threads = [threading.Thread(target=drain, args=('c1', of1), daemon=True), threading.Thread(target=drain, args=('c2', of2), daemon=True),
             threading.Thread(target=generate, daemon=True)]
  for t in threads:
    t.start()
  rc.multi_process(il, m, tf1, of1, tf2, of2, processes=1, seed=info['seed'], mode='deterministic')
  for t in threads:
    t.join(timeout=120)
  assert not errs, errs
  assert got['c1'] == H.golden_fastq('edge.c1.fq.gz') and got['c2'] == H.golden_fastq('edge.c2.fq.gz')


@pytest.mark.parametrize('level', [1, 6])
def test_gzip_sink_gunzips_to_the_plain_bytes(tmp_path, monkeypatch, level):
  """`--gzip`: multi-member gzip written by the sink's deflate threads (one member per piece) must
  gunzip to exactly the bytes of the plain run -- what `>(gzip > r1.fq.gz)` gives the reference
  (Readme.md:170).  A .gz file name switches it on by itself."""
  import gzip
  import mitty_b200.simulation.illumina as il
  import mitty_b200.simulation.readgenerate as rg
  monkeypatch.setattr(rg, 'CHUNK_BYTES', 50000)        # several members per unit
  info = H.golden()['fastq']['edge']
  wl = synth.edge_workload()
  fa, vcf, bed = synth.write_workload(wl, str(tmp_path / 'edge'))
  r1, r2 = str(tmp_path / 'r1.fq.gz'), str(tmp_path / 'r2.fq.gz')
  rg.process_multi_threaded(fa, vcf, wl['sample'], bed, il, H.model(info['model']), info['coverage'], r1, r2,
                            threads=2, seed=info['seed'], mode='deterministic', devices=[0, 0], gzip_level=level if level != 1 else None)
  raw1 = open(r1, 'rb').read()
  assert raw1[:2] == b'\x1f\x8b' and raw1.count(b'\x1f\x8b\x08') > 3
  assert gzip.open(r1, 'rb').read() == H.golden_fastq('edge.r1.fq.gz') and gzip.open(r2, 'rb').read() == H.golden_fastq('edge.r2.fq.gz')
  assert len(raw1) < 0.5 * len(H.golden_fastq('edge.r1.fq.gz'))


def test_generate_reads_without_fastq2(tmp_path):
  """`generate-reads` without --fastq2: the writer zips the template's records with the open files
  (readgenerate.py:246-248), so only file 1 is written -- with the same bytes as in a paired run
  (the qname still describes both reads)."""
  from click.testing import CliRunner
  from mitty_b200.cli import cli
  info = H.golden()['fastq']['edge']
  wl = synth.edge_workload()
  fa, vcf, bed = synth.write_workload(wl, str(tmp_path / 'edge'))
  r1 = str(tmp_path / 'only1.fq')
  res = CliRunner().invoke(cli, ['generate-reads', fa, vcf, wl['sample'], bed, info['model'], str(info['coverage']), str(info['seed']),
                                 r1, '--threads', '1', '--deterministic'], catch_exceptions=False)
  assert res.exit_code == 0, res.output
  assert open(r1, 'rb').read() == H.golden_fastq('edge.r1.fq.gz')
  assert not [x for x in os.listdir(str(tmp_path)) if x.endswith('.fq') and x != 'only1.fq']      # no second file appears
  # --deterministic with --corrupt is refused before any output is opened
  r3 = str(tmp_path / 'never.fq')
  res = CliRunner().invoke(cli, ['generate-reads', fa, vcf, wl['sample'], bed, info['model'], '30', '7', r3, '--deterministic', '--corrupt'])
  assert res.exit_code != 0 and not os.path.exists(r3)


@pytest.mark.timeout(1500)
def test_bench_unit_full_size_exact(eng):
  """ONE unit of exactly the workload bench.py's number is quoted on -- synth.chr1_shaped(seed=7,
  length=249250621), copy 1, Philox mode, perfect reads: 5.7 M templates, 2.1 GB per file (4.2 GB per
  launch), template starts near 2.5e8 -- against the oracle fed with the device's own
  draws: count and sha256 of both files.  (About 75 s of oracle time.)  The fused-corruption twin of
  the same unit is then checked against the numpy specification on a 1 % sample of its records."""
  import hashlib
  import mitty_b200.simulation.illumina as il
  from mitty_b200.engine import MODE_PHILOX
  from tests import philox_ref as PR
  wl = synth.chr1_shaped(seed=7, length=249250621, n_runs=39)
  m = H.model('hiseq-X-v2.5-Garvan.pkl')
  rm = il.read_model_params(m, 30.0)
  eng.load_model(rm)
  r = H.workload_regions(wl)[0]
  rid = eng.load_region(r['ref'], 0)
  cp = eng.build_copy(rid, r['v'][1])
  n = int((cp.p_max - cp.p_min) * rm['p'] * 1.2)
  seed = (2000 * 7919 + 2 * 104729) & 0xFFFFFFFF        # bench.py's seed of its first timed step, unit k = 2 (copy 1, pass 0)
  ts, te, fo = eng.sample_templates(n, rm['p'], MODE_PHILOX, seed, cp=cp)
  keep = te >= 0
  f1, f2, cnt, nk, nb = eng.generate_unit(cp, n, rm['p'], MODE_PHILOX, seed, '@S:0:2:', '|1|1')
  assert nb > 2000000000 and cnt > 5000000 and cnt < nk
  o1, o2, ocnt = oracle.generate_unit(r['ref'], 1, H.oracle_cv(r['v'][1]), rm['rlen'], ts[keep], te[keep], fo[keep], 'S:0:2', '1', 1,
                                      cap=int(nb) + 4096)
  assert cnt == ocnt and len(o1) == nb == f1.size
  assert hashlib.sha256(f1).hexdigest() == H.sha256(o1) and hashlib.sha256(f2).hexdigest() == H.sha256(o2)
  del o1, o2
  # fused corruption of the same unit vs the numpy specification, on every 100th record
  c1, c2, ccnt, _, cnb = eng.generate_unit(cp, n, rm['p'], MODE_PHILOX, seed, '@S:0:2:', '|1|1', corrupt=True, corrupt_seed=2000)
  assert ccnt == cnt and cnb == nb
  tables = PR.fused_tables(eng, 0)
  for perfect, corrupted, f in ((f1, c1, 0), (f2, c2, 1)):
    nl = np.flatnonzero(perfect == 10)
    assert nl.size == 4 * cnt
    starts = np.concatenate([[0], nl[3:-1:4] + 1])
    ends = nl[3::4] + 1
    pick = np.arange(0, cnt, 100)
    sample = b''.join(perfect[starts[i]:ends[i]].tobytes() for i in pick)
    want = PR.corrupt_file(sample, f, tables, 2000, seed ^ 0x636f7231, serials=pick)
    assert b''.join(corrupted[starts[i]:ends[i]].tobytes() for i in pick) == want
  eng.free_copy(cp); eng.free_region(rid)


@pytest.mark.parametrize('workers,batch', [(1, True), (4, True), (1, False), (4, False)])
def test_exome_style_bed_many_small_regions(tmp_path, workers, batch):
  """A BED of 1000 regions of 2 kb (4000 work units in the reference's shuffled schedule order,
  readgenerate.py:129-159), several host workers per GPU: deterministic mode == the oracle's
  generate-reads byte for byte, whatever the number of workers, on the batch path (one launch
  sequence for all units of a worker) and unit by unit."""
  import mitty_b200.simulation.illumina as il
  import mitty_b200.simulation.readgenerate as rg
  n_reg, width = 1000, 2000
  wl = synth.config1(contig_len=n_reg * width * 2 + 10000, names=('1',))
  wl['regions'] = [('1', 5000 + 2 * width * k, 5000 + 2 * width * k + width) for k in range(n_reg)]
  # variants whose deletions would cross a region end are not part of this test's subject
  t = wl['tables'][0]
  ends = np.array([r[2] for r in wl['regions']]); starts = np.array([r[1] for r in wl['regions']])
  j = np.searchsorted(starts, t.pos - 1, side='right') - 1
  reflen = t.ref_off[1:] - t.ref_off[:-1]
  ok = (j < 0) | (t.pos - 1 >= ends[np.maximum(j, 0)]) | (t.pos - 1 + reflen + 1 < ends[np.maximum(j, 0)])
  wl['tables'][0] = synth._subset(t, ok)
  m = H.model('hiseq-X-v2.5-Garvan.pkl')
  fa, vcf, bed = synth.write_workload(wl, str(tmp_path / 'exome'))
  r1, r2 = str(tmp_path / 'r1.fq'), str(tmp_path / 'r2.fq')
  rg.process_multi_threaded(fa, vcf, wl['sample'], bed, il, m, 30.0, r1, r2, threads=1, seed=7, mode='deterministic', workers_per_gpu=workers,
                            batch_small=batch)
  o1, o2, n = oracle.generate_reads_cmd(H.oracle_regions(H.workload_regions(wl)), m, 30.0, 7, wl['sample'])
  assert n > 150000 and rg.last_run['templates'] == n
  assert rg.last_run['batches'] == (workers if batch else 0)
  assert H.sha256(open(r1, 'rb').read()) == H.sha256(o1) and H.sha256(open(r2, 'rb').read()) == H.sha256(o2)


def _mixed_bed_workload():
  """Small regions (batch path) with two large ones in between (unit path), N runs and a soft-masked stretch."""
  wl = synth.config1(contig_len=1200000, names=('1', '2'))
  regs = []
  for c in ('1', '2'):
    regs += [(c, 3000 + 3000 * k, 3000 + 3000 * k + 1200 + 37 * (k % 7)) for k in range(120)]
    regs.append((c, 500000, 700000))
    regs += [(c, 800000 + 2500 * k, 800000 + 2500 * k + 900) for k in range(100)]
  wl['regions'] = regs
  for i, (name, seq) in enumerate(wl['contigs']):
    seq = np.array(seq, copy=True)
    seq[3100:3130] = ord('N'); seq[6200] = ord('R'); seq[9000:9400] |= 0x20; seq[805000:805020] = ord('N')
    wl['contigs'][i] = (name, seq)
  for i, t in enumerate(wl['tables']):
    starts = np.array(sorted(r[1] for r in regs if r[0] == wl['contigs'][i][0])); ends = np.array(sorted(r[2] for r in regs if r[0] == wl['contigs'][i][0]))
    j = np.searchsorted(starts, t.pos - 1, side='right') - 1
    reflen = t.ref_off[1:] - t.ref_off[:-1]
    ok = (j < 0) | (t.pos - 1 >= ends[np.maximum(j, 0)]) | (t.pos - 1 + reflen + 1 < ends[np.maximum(j, 0)])
    wl['tables'][i] = synth._subset(t, ok)
  return wl


@pytest.mark.parametrize('corrupt', [False, True])
def test_batch_path_equals_unit_path(tmp_path, corrupt):
  """Production mode (Philox, with and without fused corruption) on a BED that mixes small and large regions:
  the batch path, unit by unit, three workers, gzip members and FIFOs (sequential targets) all give the
  same bytes; and every perfect read passes the god-aligner round trip."""
  import gzip
  import mitty_b200.simulation.illumina as il
  import mitty_b200.simulation.readgenerate as rg
  wl = _mixed_bed_workload()
  m = H.model('hiseq-X-v2.5-Garvan.pkl')
  fa, vcf, bed = synth.write_workload(wl, str(tmp_path / 'mix'))
  out = {}
  for tag, kw in (('unit', dict(batch_small=False)), ('batch', dict()), ('batch3', dict(workers_per_gpu=3)),
                  ('gz', dict(gzip_level=1)), ('pwrite_off', dict(sink_threads=1))):
    r1, r2 = str(tmp_path / (tag + '1.fq')), str(tmp_path / (tag + '2.fq'))
    rg.process_multi_threaded(fa, vcf, wl['sample'], bed, il, m, 30.0, r1, r2, threads=1, seed=11, mode='philox', corrupt=corrupt, **kw)
    rd = (lambda p: gzip.open(p, 'rb').read()) if tag == 'gz' else (lambda p: open(p, 'rb').read())
    out[tag] = (H.sha256(rd(r1)), H.sha256(rd(r2)), rg.last_run['templates'], rg.last_run['batches'])
  assert out['unit'][3] == 0 and out['batch'][3] >= 2 and out['batch3'][3] >= 3
  assert out['unit'][2] > 30000
  for tag in ('batch', 'batch3', 'gz', 'pwrite_off'):
    assert out[tag][:3] == out['unit'][:3], tag
  # sequential targets (FIFOs): pieces that run through several units are appended in order
  import threading
  f1, f2 = str(tmp_path / 'p1'), str(tmp_path / 'p2')
  os.mkfifo(f1); os.mkfifo(f2)
  got = {}

  def drain(name, path):
    with open(path, 'rb') as fp:
      got[name] = H.sha256(fp.read())
  th = [threading.Thread(target=drain, args=(1, f1), daemon=True), threading.Thread(target=drain, args=(2, f2), daemon=True)]
  for t in th:
    t.start()
  rg.process_multi_threaded(fa, vcf, wl['sample'], bed, il, m, 30.0, f1, f2, threads=1, seed=11, mode='philox', corrupt=corrupt, workers_per_gpu=2)
  for t in th:
    t.join(timeout=120)
  assert (got[1], got[2]) == out['unit'][:2]
  if not corrupt:   # every read of the batch path's files is where its qname says (god-aligner round trip on the device)
    from mitty_b200.simulation.readcheck import check_fastq
    res = check_fastq(fa, vcf, wl['sample'], bed, str(tmp_path / 'batch1.fq'), str(tmp_path / 'batch2.fq'))
    assert res['templates'] == out['unit'][2] and res['bad'] == 0, res['examples']
