"""Production (Philox) mode on the GPU: exactness of the emit path given the device's own template
draws, god-aligner round trips, and statistical equivalence with the reference / the model."""
import os

import numpy as np
import pytest
from scipy import stats

import oracle
from mitty_b200 import synth
from tests import helpers as H
from tests.test_gpu_parity import gpu_generate

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def eng():
  from mitty_b200.engine import Engine
  e = Engine(0)
  yield e
  e.close()


def test_philox_units_exact_vs_oracle(eng):
  """The device's Philox template draws are read back (mg_sample_templates) and handed to the
  oracle: the unit's FASTQ must then agree byte for byte (scan, compaction, serials, file order)."""
  import mitty_b200.simulation.illumina as il
  from mitty_b200.engine import MODE_PHILOX
  wl = synth.config1(contig_len=300000)
  m = H.model('hiseq-X-v2.5-Garvan.pkl')
  rm = il.read_model_params(m, 30.0)
  eng.load_model(rm)
  for ri, r in enumerate(H.workload_regions(wl)):
    rid = eng.load_region(r['ref'], r['region'][1])
    for cpy, vl in enumerate(r['v']):
      cp = eng.build_copy(rid, vl)
      n = int((cp.p_max - cp.p_min) * rm['p'] * 1.2)
      seed = 1000 * ri + cpy
      ts, te, fo = eng.sample_templates(n, rm['p'], MODE_PHILOX, seed, cp=cp)
      keep = te >= 0
      assert 0.75 < keep.mean() < 0.92          # the 1.2x over-draw: ~1/1.2 of the candidates fit
      assert np.unique(ts).size == n            # the Feistel shuffle is a permutation of distinct starts
      f1, f2, cnt, nk, nb = eng.generate_unit(cp, n, rm['p'], MODE_PHILOX, seed, '@S:0:{}:'.format(ri), '|{}|{}'.format(r['region'][0], cpy))
      assert nk == keep.sum()
      o1, o2, ocnt = oracle.generate_unit(r['ref'], r['region'][1] + 1, H.oracle_cv(vl), rm['rlen'], ts[keep], te[keep], fo[keep],
                                          'S:0:{}'.format(ri), r['region'][0], cpy)
      assert cnt == ocnt
      assert f1.tobytes() == o1 and f2.tobytes() == o2
      eng.free_copy(cp)
    eng.free_region(rid)


def test_philox_roundtrip_and_coverage(eng):
  """Every read of a Philox-mode run re-derives from its qname (god-aligner contract), and the
  coverage / template-length statistics match the reference run of the same workload."""
  import mitty_b200.simulation.readgenerate as rg
  wl = synth.config1(contig_len=100000)
  m = H.model('hiseq-X-v2.5-Garvan.pkl')
  regs = H.workload_regions(wl)
  f1, f2, n = gpu_generate(eng, wl, m, 30.0, 7, 'philox', regions=regs)
  gold = H.golden()['fastq']['mid']
  assert abs(n - gold['pairs']) < 5 * np.sqrt(gold['pairs'])
  idx = {}
  def index_for(chrom, cpy):
    if (chrom, cpy) not in idx:
      r = next(r for r in regs if r['region'][0] == chrom)
      idx[(chrom, cpy)] = H.HaplotypeIndex(r['ref'], r['region'][1] + 1, H.oracle_cv(r['v'][cpy]))
    return idx[(chrom, cpy)]
  checked, errs = H.roundtrip_fastq(f1, f2, index_for)
  assert checked == 2 * n and not errs, errs[:3]
  # coverage histogram of template starts on contig '1' vs the reference's (KS on the binned CDFs)
  starts, tlens = [], []
  for line in f1.decode().split('\n')[0::4]:
    if not line:
      continue
    a, b = rg.parse_qname(line[1:])
    if a.chrom == '1':
      starts.append(min(a.pos, b.pos)); tlens.append(max(a.pos, b.pos) + 150 - min(a.pos, b.pos))
  ref_hist = np.load(os.path.join(H.GOLDEN, 'mid_coverage.npz'))['hist']
  got_hist = np.histogram(starts, bins=100, range=(0, 100000))[0]
  assert stats.chisquare(got_hist[1:-1] * (ref_hist[1:-1].sum() / got_hist[1:-1].sum()), ref_hist[1:-1]).pvalue > 0.01 or \
    stats.ks_2samp(np.repeat(np.arange(100), got_hist), np.repeat(np.arange(100), ref_hist)).pvalue > 0.01
  # template lengths follow the model's empirical distribution
  pm = np.diff(np.concatenate([[0.0], m['cum_tlen']]))
  tl = np.array(tlens)
  tl = tl[tl > 150]
  lo, hi = 151, 999
  obs = np.bincount(tl, minlength=1001)[lo:hi + 1].astype(float)
  exp = pm[lo:hi + 1] / pm[lo:hi + 1].sum() * obs.sum()
  big = exp > 5
  assert stats.chisquare(obs[big] * (exp[big].sum() / obs[big].sum()), exp[big]).pvalue > 0.01


def _bq_stats(c, r, rlen):
  hist = np.zeros((rlen, 94)); sub = np.zeros(rlen)
  lc, lr = c.decode().split('\n'), r.decode().split('\n')
  for k in range(0, len(lc) - 1, 4):
    q = np.frombuffer(lc[k + 3].encode(), dtype=np.uint8) - 33
    hist[np.arange(q.size), q] += 1
    sub += np.frombuffer(lc[k + 1].encode(), dtype=np.uint8) != np.frombuffer(lr[k + 1].encode(), dtype=np.uint8)
  return hist, sub


@pytest.mark.parametrize('fused', [False, True])
def test_philox_corruption_statistics(eng, fused):
  """Per-cycle base-quality and substitution-rate distributions of Philox corruption vs the model
  (exact expectation) and vs the reference's own corrupt-reads run (golden counts): p > 0.01."""
  from mitty_b200.engine import MODE_PHILOX
  wl = synth.config1(contig_len=100000)
  m = H.model('hiseq-X-v2.5-Garvan.pkl')
  regs = H.workload_regions(wl)
  p1, p2, n = gpu_generate(eng, wl, m, 30.0, 7, 'philox', regions=regs)
  if fused:
    c1, c2, n2 = gpu_generate(eng, wl, m, 30.0, 7, 'philox', corrupt=True, regions=regs)
    assert n2 == n
  else:
    eng.load_model(m)
    c1, c2, n2 = eng.corrupt_fastq(p1, p2, mode=MODE_PHILOX, seed=11)
    c1, c2 = c1.tobytes(), c2.tobytes()
    assert n2 == n
  # records keep their layout: same qnames, same lengths
  assert len(c1) == len(p1) and c1.split(b'\n')[0::4] == p1.split(b'\n')[0::4]
  gold = np.load(os.path.join(H.GOLDEN, 'mid_corrupt_stats.npz'))
  pvals_model, pvals_ref = [], []
  for mate, (c, r) in enumerate(((c1, p1), (c2, p2))):
    hist, sub = _bq_stats(c, r, 150)
    pm = np.diff(np.concatenate([np.zeros((150, 1)), m['cum_bq_mat'][mate, :150, :]], axis=1), axis=1)
    exp_sub = (pm * oracle.PHRED_P[:94]).sum(axis=1) * n
    for cyc in range(0, 150, 7):
      # vs the model's exact per-cycle distribution (cells with a healthy expectation, rest pooled)
      big = pm[cyc] * n > 20
      obs = np.append(hist[cyc][big], hist[cyc][~big].sum()); exp = np.append(pm[cyc][big], pm[cyc][~big].sum()) * n
      keep = exp > 0
      pvals_model.append(stats.chisquare(obs[keep], exp[keep] * (obs[keep].sum() / exp[keep].sum())).pvalue)
      # vs the reference's own corrupt-reads sample of the same workload: two-sample KS on the BQ values
      a, b = hist[cyc].astype(np.int64), gold['bq_hist'][mate, cyc].astype(np.int64)
      pvals_ref.append(stats.ks_2samp(np.repeat(np.arange(94), a), np.repeat(np.arange(94), b)).pvalue)
    # substitutions: a Poisson count with the model's expectation, and vs the reference's count
    z = (sub.sum() - exp_sub.sum()) / np.sqrt(exp_sub.sum())
    assert abs(z) < 4, (sub.sum(), exp_sub.sum())
    zr = (sub.sum() - gold['sub_count'][mate].sum() * n / float(gold['pairs'])) / np.sqrt(2 * sub.sum())
    assert abs(zr) < 4
    # per-cycle error-rate profile vs the reference's (KS over cycles weighted by substitution counts)
    assert stats.ks_2samp(np.repeat(np.arange(150), sub.astype(np.int64)),
                          np.repeat(np.arange(150), gold['sub_count'][mate].astype(np.int64))).pvalue > 0.01
  # the distributions are EXACTLY specified and tested bit for bit elsewhere
  # (test_philox_corruption_exact_vs_numpy_spec); here every per-cycle test must clear p > 0.01
  # after Bonferroni correction for the number of cycles tested, and low p-values must be rare
  for pv in (pvals_model, pvals_ref):
    assert min(pv) > 0.01 / len(pv), sorted(pv)[:5]
    assert np.mean(np.array(pv) < 0.01) < 0.1, sorted(pv)[:5]


def test_philox_large_unit_exact(eng):
  """A 20 Mb contig with GRCh37-like N runs (the > 2 N template drop fires): one Philox unit,
  ~0.5 M templates, checked byte for byte against the oracle fed with the device's draws."""
  import mitty_b200.simulation.illumina as il
  from mitty_b200.engine import MODE_PHILOX
  wl = synth.chr1_shaped(seed=5, length=20000000, n_runs=9)
  m = H.model('hiseq-X-v2.5-Garvan.pkl')
  rm = il.read_model_params(m, 30.0)
  eng.load_model(rm)
  r = H.workload_regions(wl)[0]
  rid = eng.load_region(r['ref'], 0)
  cp = eng.build_copy(rid, r['v'][1])
  n = int((cp.p_max - cp.p_min) * rm['p'] * 1.2)
  ts, te, fo = eng.sample_templates(n, rm['p'], MODE_PHILOX, 99, cp=cp)
  keep = te >= 0
  f1, f2, cnt, nk, nb = eng.generate_unit(cp, n, rm['p'], MODE_PHILOX, 99, '@BIG:0:0:', '|1|1')
  o1, o2, ocnt = oracle.generate_unit(r['ref'], 1, H.oracle_cv(r['v'][1]), rm['rlen'], ts[keep], te[keep], fo[keep], 'BIG:0:0', '1', 1)
  assert cnt == ocnt and cnt < nk      # some templates were dropped for N content
  assert H.sha256(f1.tobytes()) == H.sha256(o1) and H.sha256(f2.tobytes()) == H.sha256(o2)
  eng.free_copy(cp); eng.free_region(rid)


@pytest.mark.parametrize('wl_fn,cpy,model_name', [(synth.edge_workload, 1, 'hiseq-X-v2.5-Garvan.pkl'),
                                                  (synth.softmask_workload, 0, 'hiseq-X-v2.5-Garvan.pkl'),
                                                  (synth.edge_workload, 0, '1kg-pcr-free.pkl'),   # 2x250: the wide register window, 256-entry rows
                                                  (synth.edge_workload, 1, 'hiseq-2500-v1-pcr-free.pkl'),
                                                  (synth.edge_workload, 1, 'hiseq-X-v2.5-Garvan.pkl:200'),   # reads longer than max_rlen: BQ 93, 9-bit codes
                                                  (synth.edge_workload, 1, 'hiseq-X-v2.5-Garvan.pkl:161'),   # both sides of the first register-window switch
                                                  (synth.edge_workload, 1, 'hiseq-X-v2.5-Garvan.pkl:162'),
                                                  (synth.edge_workload, 1, 'hiseq-X-v2.5-Garvan.pkl:300')])   # the wide window at the model's last cycle
def test_philox_corruption_exact_vs_numpy_spec(eng, wl_fn, cpy, model_name):
  """Production-mode corruption is fully specified (Philox counters, one joint alias row per (mate,
  cycle)): the fused emit kernel and the standalone corrupt kernel must reproduce the numpy
  restatement of that specification byte for byte, and the tables the library builds at load time
  must equal the Python restatement of Vose's method."""
  import mitty_b200.simulation.illumina as il
  from mitty_b200.engine import MODE_PHILOX
  from tests import philox_ref as PR
  m = dict(H.model(model_name.split(':')[0]))
  if ':' in model_name:
    m['mean_rlen'] = int(model_name.split(':')[1])       # legal: the path reads only mean_rlen (illumina.py:20)
  rm = il.read_model_params(m, 30.0)
  eng.load_model(rm)
  tabs = []
  for which, rows in ((0, int(rm['rlen'])), (1, m['cum_bq_mat'].shape[1])):
    alias, ks, c9 = eng.model_tables(which)
    assert (ks, c9) == PR.table_shape(m['cum_bq_mat'], oracle.PHRED_P, rows)
    np.testing.assert_array_equal(alias, PR.joint_tables(m['cum_bq_mat'], oracle.PHRED_P, ks, c9, n_rows=rows))
    tabs.append((alias, ks, c9))
  assert tabs[1][2] == 1                                 # the rows beyond max_rlen are quality 93
  if ':' in model_name:
    assert tabs[0][2] == 1
  r = H.workload_regions(wl_fn())[0]
  rid = eng.load_region(r['ref'], r['region'][1])
  cp = eng.build_copy(rid, r['v'][cpy])
  n = int((cp.p_max - cp.p_min) * 0.1)
  unit_seed, cseed = 4242, 77
  p1, p2, cnt, _, _ = eng.generate_unit(cp, n, 0.1, MODE_PHILOX, unit_seed, '@E:0:0:', '|e|1')
  c1, c2, ccnt, _, _ = eng.generate_unit(cp, n, 0.1, MODE_PHILOX, unit_seed, '@E:0:0:', '|e|1', corrupt=True, corrupt_seed=cseed)
  assert cnt == ccnt and cnt > 500
  k1 = unit_seed ^ 0x636f7231
  assert c1.tobytes() == PR.corrupt_file(p1.tobytes(), 0, tabs[0], cseed, k1)
  assert c2.tobytes() == PR.corrupt_file(p2.tobytes(), 1, tabs[0], cseed, k1)
  # standalone corrupt-reads over the same perfect reads
  eng.load_model(m)
  s1, s2, scnt = eng.corrupt_fastq(p1, p2, mode=MODE_PHILOX, seed=cseed)
  assert scnt == cnt
  assert s1.tobytes() == PR.corrupt_file(p1.tobytes(), 0, tabs[1], cseed, 0x636f7232)
  assert s2.tobytes() == PR.corrupt_file(p2.tobytes(), 1, tabs[1], cseed, 0x636f7232)
  eng.free_copy(cp); eng.free_region(rid)


def test_philox_full_size_properties(eng):
  """BASELINE-scale unit (a 60 Mb contig with N runs, ~1.5 M templates, fused corruption), checked
  through size-independent properties: run-to-run determinism, record structure, consecutive
  serials, the N filter, and god-aligner round trips of a random sample of the PERFECT twin run
  (same seeds, so the same templates)."""
  import mitty_b200.simulation.illumina as il
  import mitty_b200.simulation.readgenerate as rg
  from mitty_b200.engine import MODE_PHILOX
  wl = synth.chr1_shaped(seed=3, length=60000000, n_runs=12)
  m = H.model('hiseq-X-v2.5-Garvan.pkl')
  rm = il.read_model_params(m, 30.0)
  eng.load_model(rm)
  r = H.workload_regions(wl)[0]
  rid = eng.load_region(r['ref'], 0)
  cp = eng.build_copy(rid, r['v'][0])
  n = int((cp.p_max - cp.p_min) * rm['p'] * 1.2)
  args = (cp, n, rm['p'], MODE_PHILOX, 4242, '@BIG:0:0:', '|1|0')
  c1, c2, cnt, nk, nb = eng.generate_unit(*args, corrupt=True, corrupt_seed=9)
  assert cnt > 1200000 and cnt < nk
  sha = (H.sha256(c1.tobytes()), H.sha256(c2.tobytes()))
  d1, d2, cnt2, _, _ = eng.generate_unit(*args, corrupt=True, corrupt_seed=9)
  assert cnt2 == cnt and (H.sha256(d1.tobytes()), H.sha256(d2.tobytes())) == sha      # deterministic
  p1, p2, cntp, _, _ = eng.generate_unit(*args)                                         # perfect twin
  assert cntp == cnt and p1.size == c1.size
  for a, b in ((c1, p1), (c2, p2)):
    nl = np.flatnonzero(a == 10)
    assert nl.size == 4 * cnt and np.array_equal(nl, np.flatnonzero(b == 10))            # same layout
    starts = np.concatenate([[0], nl[3:-1:4] + 1])
    assert (a[starts] == ord('@')).all() and (a[nl[1::4] + 1] == ord('+')).all()
    assert ((nl[1::4] - nl[0::4] - 1) == 150).all() and ((nl[3::4] - nl[2::4] - 1) == 150).all()
    # qname lines are identical in the corrupted and the perfect file; qualities are in range
    k = np.random.RandomState(1).randint(0, cnt, size=2000)
    for i in k[:200]:
      assert a[starts[i]:nl[4 * i]].tobytes() == b[starts[i]:nl[4 * i]].tobytes()
    q = np.concatenate([a[nl[4 * i + 2] + 1:nl[4 * i + 3]] for i in k])
    assert q.min() >= 33 + 1 and q.max() <= 33 + 41
  # serials are 1..cnt in file order
  nl = np.flatnonzero(p1 == 10)
  starts = np.concatenate([[0], nl[3:-1:4] + 1])
  for i in (0, 1, 9, 10, 99999, 100000, cnt - 1):
    assert p1[starts[i]:nl[4 * i]].tobytes().split(b'|')[0] == '@BIG:0:0:{}'.format(i + 1).encode()
  # no read with more than two N; sampled round trips through the qname
  idx = H.HaplotypeIndex(r['ref'], 1, H.oracle_cv(r['v'][0]))
  rs = np.random.RandomState(2)
  errs = []
  for which, buf in ((0, p1), (1, p2)):
    nlb = np.flatnonzero(buf == 10)
    st = np.concatenate([[0], nlb[3:-1:4] + 1])
    for i in rs.randint(0, cnt, size=4000):
      qn = buf[st[i] + 1:nlb[4 * i]].tobytes().decode()
      seq = buf[nlb[4 * i] + 1:nlb[4 * i + 1]].tobytes().decode()
      assert seq.count('N') <= 2
      e = idx.check(rg.parse_qname(qn)[which], seq)
      if e:
        errs.append((qn, e))
  assert not errs, errs[:3]
  eng.free_copy(cp); eng.free_region(rid)
