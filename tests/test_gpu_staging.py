"""GPU tests of the rare paths of the emit, corrupt and plan kernels, each against the references the rest
of the suite trusts (the oracle for perfect reads, tests/philox_ref.py for Philox corruption):

- k_unit_emit's warp tiles that do not fit the shared-memory stage in one batch (long qname strings, long
  reads), records larger than the whole stage (emit_oversize), units over many variant nodes, and the
  relaunch after the output outgrew its estimate;
- k_unit_plan's tile protocol at tile-count edges, over long runs of tiles with nothing kept and tiles
  that only the N filter empties;
- production-mode corrupt-reads on ragged lengths, odd names and comments, long names that split the
  staged kernel's batches, and a name long enough to send the call to k_corrupt.

Every file is compared byte for byte; coverage guards assert that the inputs really reach the path a test
is named after, so a change to a stage size cannot make a test hollow unnoticed."""
import re

import numpy as np
import pytest

import oracle
from mitty_b200 import synth
from mitty_b200.lib import vcfio
from tests import helpers as H
from tests import philox_ref as PR

pytestmark = pytest.mark.gpu

QN_MAX = 192            # MG_QN_MAX (mg_internal.h): longest qname prefix / mid string
PLAN_TILE = 256         # MG_PLAN_TILE (mg_internal.h): candidates per tile of k_unit_plan
EMIT_KEY = 0x636f7231   # fused corruption key: unit seed ^ this (mg_unit_generate)
CORRUPT_KEY = 0x636f7232


@pytest.fixture(scope='module')
def eng():
  from mitty_b200.engine import Engine
  e = Engine(0)
  yield e
  e.close()


# ---- the emit kernel's stage, restated ---------------------------------------------------------------

def stage_cap(L):
  """Bytes of a warp's stage in k_unit_emit: 32 records with an average qname, at most 48 KB, a multiple
  of 16 (unit_generate in mg_api.cu)."""
  return min(32 * (2 * L + 5 + 96), 48 * 1024) & ~15


def record_bounds(buf):
  """-> (start, end) byte offsets of the 4-line records of a FASTQ buffer."""
  nl = np.flatnonzero(np.frombuffer(buf, dtype=np.uint8) == 10)
  ends = nl[3::4] + 1
  return np.concatenate([[0], ends[:-1]]).astype(np.int64), ends.astype(np.int64)


def stage_batches(starts, ends, cap):
  """How k_unit_emit (mg_kernels.cu) emits each warp tile of 32 records: from the first record lo not yet
  emitted, a batch takes the records whose end e fits, e - start[lo] + (start[lo] & 15) <= cap (the stage
  keeps the output's 16-byte phase).  A record that does not fit alone goes straight to global memory
  (emit_oversize).  -> per tile a list of (records, oversize) batches."""
  tiles = []
  for t0 in range(0, starts.size, 32):
    t1 = min(t0 + 32, starts.size)
    lo, tile = t0, []
    while lo < t1:
      goff = int(starts[lo])
      pad = goff & 15
      hi = lo
      while hi < t1 and int(ends[hi]) - goff + pad <= cap:
        hi += 1
      tile.append((max(hi, lo + 1) - lo, hi == lo))
      lo = max(hi, lo + 1)
    tiles.append(tile)
  return tiles


def check_tile_splits(buf, L, min_ways):
  """Coverage guard of the batch-splitting loop: most full warp tiles of buf are emitted in several
  batches, and some in at least min_ways."""
  tiles = stage_batches(*record_bounds(buf), stage_cap(L))
  full = [len(t) for t in tiles if sum(b[0] for b in t) == 32]
  assert full and np.mean(np.array(full) > 1) > 0.5, (L, full[:20])
  assert max(full) >= min_ways, (L, max(full))


def synth_model(n_cycles, seed=0):
  """A small read model for any read length: the template lengths of hiseq-X-v2.5-Garvan and, per mate
  and cycle, three qualities (so each joint alias row has 12 outcomes)."""
  rs = np.random.RandomState(seed)
  n_bq = 41
  qa = rs.randint(10, 20, size=(2, n_cycles, 1))
  qb = rs.randint(25, 35, size=(2, n_cycles, 1))
  wa = rs.uniform(0.05, 0.3, size=(2, n_cycles, 1))
  wb = rs.uniform(0.2, 0.5, size=(2, n_cycles, 1))
  b = np.arange(n_bq)[None, None, :]
  cum = (b >= qa) * wa + (b >= qb) * wb + (b >= 40) * (1.0 - wa - wb)
  return {'cum_tlen': H.model('hiseq-X-v2.5-Garvan.pkl')['cum_tlen'], 'cum_bq_mat': cum, 'rlen': n_cycles}


def fused_tables(eng, m, rows=40):
  """The emit kernel's alias tables as the library built them, with their first rows pinned against the
  Python restatement of Vose's method."""
  alias, ks, c9 = eng.model_tables(0)
  head = np.ascontiguousarray(m['cum_bq_mat'][:, :rows])
  assert (ks, c9) == PR.table_shape(head, oracle.PHRED_P, rows)
  np.testing.assert_array_equal(alias[:, :rows], PR.joint_tables(head, oracle.PHRED_P, ks, c9))
  return alias, ks, c9


def philox_unit_checks(eng, cp, ref, start1, cv, L, n, p, seed, prefix, mid, stub, chrom, cpy, tables, cseed=77):
  """One Philox unit: perfect reads == the oracle fed with the device's own draws, fused corruption ==
  the numpy specification on the perfect twin.  -> perfect file 1 (bytes)."""
  from mitty_b200.engine import MODE_PHILOX
  ts, te, fo = eng.sample_templates(n, p, MODE_PHILOX, seed, cp=cp)
  keep = te >= 0
  p1, p2, cnt, nk, _ = eng.generate_unit(cp, n, p, MODE_PHILOX, seed, prefix, mid)
  assert nk == keep.sum()
  o1, o2, ocnt = oracle.generate_unit(ref, start1, cv, L, ts[keep], te[keep], fo[keep], stub, chrom, cpy)
  assert cnt == ocnt and cnt > 0
  assert p1.tobytes() == o1 and p2.tobytes() == o2
  c1, c2, ccnt, _, _ = eng.generate_unit(cp, n, p, MODE_PHILOX, seed, prefix, mid, corrupt=True, corrupt_seed=cseed)
  assert ccnt == cnt
  assert c1.tobytes() == PR.corrupt_file(o1, 0, tables, cseed, seed ^ EMIT_KEY)
  assert c2.tobytes() == PR.corrupt_file(o2, 1, tables, cseed, seed ^ EMIT_KEY)
  return o1


# ---- 1. long qname strings on the unit path ---------------------------------------------------------

# (sample, chromosome): '@' + sample + ':0:0:' and '|' + chromosome + '|' + copy are 192 bytes, or about 100
LONG_NAMES = {'max': ('S' * (QN_MAX - 6), 'c' * (QN_MAX - 3)), 'mid': ('s' * 94, 'chr' + 'x' * 95)}


@pytest.mark.parametrize('names', ['max', 'mid'])
@pytest.mark.parametrize('L', [1, 16, 150, 250])
def test_long_qnames_explicit(eng, L, names):
  """Explicit templates on the edge workload with the longest qname strings the product accepts: the
  warp tiles no longer fit the stage in one batch."""
  from mitty_b200.engine import MODE_EXPLICIT
  sample, chrom = LONG_NAMES[names]
  regs = H.workload_regions(synth.edge_workload())[:3]
  rs = np.random.RandomState(L)
  eng.load_model({'cum_tlen': np.array([1.0]), 'cum_bq_mat': np.ones((2, 300, 94)), 'rlen': L})
  perfect = []
  for r in regs:
    rid = eng.load_region(r['ref'], r['region'][1])
    for cpy, vl in enumerate(r['v']):
      cp = eng.build_copy(rid, vl)
      n = 2000
      ts = rs.randint(cp.p_min - 2, cp.p_max, size=n).astype(np.int64)
      tl = rs.randint(0, 3 * L + 40, size=n).astype(np.int64)
      fo = rs.randint(0, 2, size=n).astype(np.int8)
      prefix, mid = '@{}:0:0:'.format(sample), '|{}|{}'.format(chrom, cpy)
      if names == 'max':
        assert len(prefix) == len(mid) == QN_MAX
      f1, f2, cnt, nk, _ = eng.generate_unit(cp, n, 0.5, MODE_EXPLICIT, 0, prefix, mid, ts=ts, tl=tl, fo=fo)
      te = ts + np.maximum(tl, L)
      keep = (te < cp.p_max) & (ts >= cp.p_min)
      assert nk == keep.sum()
      o1, o2, ocnt = oracle.generate_unit(r['ref'], r['region'][1] + 1, H.oracle_cv(vl), L, ts[keep], te[keep], fo[:keep.sum()],
                                          '{}:0:0'.format(sample), chrom, cpy)
      assert cnt == ocnt
      assert f1.tobytes() == o1 and f2.tobytes() == o2
      perfect.append(o1)
      eng.free_copy(cp)
    eng.free_region(rid)
  for buf in perfect:
    if buf.count(b'\n') >= 4 * 32 * 8:
      check_tile_splits(buf, L, 3 if L <= 16 else 2)


@pytest.mark.parametrize('names', ['max', 'mid'])
@pytest.mark.parametrize('L', [1, 16, 150, 250])
def test_long_qnames_fused_philox(eng, L, names):
  """The same names through Philox sampling and fused corruption (hiseq-X-v2.5-Garvan with rlen = L)."""
  import mitty_b200.simulation.illumina as il
  sample, chrom = LONG_NAMES[names]
  m = dict(H.model('hiseq-X-v2.5-Garvan.pkl'))
  m['mean_rlen'] = L
  eng.load_model(il.read_model_params(m, 30.0))
  tables = eng.model_tables(0)
  r = H.workload_regions(synth.edge_workload())[0]
  rid = eng.load_region(r['ref'], r['region'][1])
  cp = eng.build_copy(rid, r['v'][1])
  n = int((cp.p_max - cp.p_min) * 0.1)
  o1 = philox_unit_checks(eng, cp, r['ref'], r['region'][1] + 1, H.oracle_cv(r['v'][1]), L, n, 0.1, 4242,
                          '@{}:0:0:'.format(sample), '|{}|1'.format(chrom), '{}:0:0'.format(sample), chrom, 1, tables)
  check_tile_splits(o1, L, 3 if L <= 16 else 2)
  eng.free_copy(cp); eng.free_region(rid)


def test_qname_strings_over_192_bytes_are_rejected(eng):
  from mitty_b200.engine import MODE_EXPLICIT
  eng.load_model({'cum_tlen': np.array([1.0]), 'cum_bq_mat': np.ones((2, 300, 94)), 'rlen': 10})
  rid = eng.load_region(np.frombuffer(H.TINY_SEQ.encode(), dtype=np.uint8), 0)
  cp = eng.build_copy(rid, vcfio.VariantList.from_variants([]))
  args = dict(ts=np.array([3], np.int64), tl=np.array([12], np.int64), fo=np.ones(1, np.int8))
  ok = '@' + 'a' * (QN_MAX - 1)
  f1, _, cnt, _, _ = eng.generate_unit(cp, 1, 0.5, MODE_EXPLICIT, 0, ok, '|' + 'b' * (QN_MAX - 1), **args)
  assert cnt == 1 and f1.tobytes().startswith((ok + '1|' + 'b' * (QN_MAX - 1) + '|').encode())
  for prefix, mid in ((ok + 'a', '|1|0'), ('@s:0:0:', '|' + 'b' * QN_MAX)):
    with pytest.raises(ValueError):
      eng.generate_unit(cp, 1, 0.5, MODE_EXPLICIT, 0, prefix, mid, **args)
  eng.free_copy(cp); eng.free_region(rid)


# ---- 3. long reads: split tiles, records at the stage size, all-oversize tiles ------------------------

@pytest.fixture(scope='module')
def long_contig():
  return synth.synth_contig(1500000, seed=41)


MIXED_L = 24540     # 2 L + 5 + qname sits at the 48 KB stage: the 16-byte phase decides stage or emit_oversize


@pytest.mark.parametrize('L', [305, 306, 800, MIXED_L, 30000])
def test_long_reads_philox(eng, long_contig, L):
  """Reads on both sides of the last register-window switch (305 / 306) and long reads that split every
  warp tile (800), sit at the stage size (MIXED_L) or exceed it (30000): perfect == oracle, fused == spec."""
  m = synth_model(L, seed=L)
  eng.load_model(m)
  tables = fused_tables(eng, m)
  rid = eng.load_region(long_contig, 0)
  cp = eng.build_copy(rid, vcfio.VariantList.from_variants([]))
  n = 2000 if L <= 1000 else 300
  p = n / (0.9 * (cp.p_max - cp.p_min))
  o1 = philox_unit_checks(eng, cp, long_contig, 1, H.oracle_cv(vcfio.VariantList.from_variants([])), L, n, p, 1000 + L,
                          '@LR:0:0:', '|lr|0', 'LR:0:0', 'lr', 0, tables)
  tiles = stage_batches(*record_bounds(o1), stage_cap(L))
  over = [[b[1] for b in t] for t in tiles]
  if L == 800:
    assert all(len(t) > 1 for t in tiles if sum(b[0] for b in t) == 32)
    assert not any(any(o) for o in over)
  elif L == MIXED_L:
    assert stage_cap(L) == 48 * 1024
    assert any(any(o) and not all(o) for o in over)          # staged and oversize records in one warp tile
  elif L == 30000:
    assert all(all(o) for o in over)
  eng.free_copy(cp); eng.free_region(rid)


# ---- 4. reads over many nodes -----------------------------------------------------------------------

@pytest.mark.parametrize('seed', [2, 3])
@pytest.mark.parametrize('model_name', ['hiseq-X-v2.5-Garvan.pkl', '1kg-pcr-free.pkl'])   # L = 150, 250
def test_reads_over_dense_variants(eng, seed, model_name):
  """Units over the variant sets of test_device_walk_dense_overlapping_variants (long deletions, stacked
  records, IUPAC ALTs): most reads leave the kernel's three-node fast path and their long CIGAR / v_list
  tokens make record sizes, and so batch bounds, irregular."""
  from mitty_b200.simulation.readgenerate import parse_qname
  m = H.model(model_name)
  L = int(m['mean_rlen'])
  eng.load_model({'cum_tlen': m['cum_tlen'], 'cum_bq_mat': m['cum_bq_mat'], 'rlen': L})
  region, bed_start, vl, _ = H.dense_variant_region(seed, alt_n=False)
  rid = eng.load_region(region, bed_start)
  cp = eng.build_copy(rid, vl)
  n = int((cp.p_max - cp.p_min) * 0.5)
  o1 = philox_unit_checks(eng, cp, region, bed_start + 1, H.oracle_cv(vl), L, n, 0.5, 31 * seed, '@D:0:0:', '|d|0', 'D:0:0', 'd', 0,
                          eng.model_tables(0))
  heads = o1.decode().split('\n')[0::4][:-1]
  ops = [len(re.findall(r'\d+[=XID]', parse_qname(h[1:])[0].cigar or '')) for h in heads]
  assert np.mean(np.array(ops) > 3) > 0.3, sorted(ops)[-10:]                  # reads over more than three nodes
  st, en = record_bounds(o1)
  assert np.unique(en - st).size > 50                                         # irregular record sizes
  eng.free_copy(cp); eng.free_region(rid)


# ---- 5. output regrow --------------------------------------------------------------------------------

def test_output_regrow_relaunches_emit():
  """Every candidate kept, long records (dense variants, 192-byte names): the unit outgrows the device
  output estimate, the first emit launch stops, the buffer is regrown and the kernel runs again.  A fresh
  engine, so no buffer left by an earlier unit is large enough already."""
  from mitty_b200.engine import Engine, MODE_EXPLICIT
  e = Engine(0)
  try:
    L = 250
    e.load_model({'cum_tlen': np.array([1.0]), 'cum_bq_mat': np.ones((2, 300, 94)), 'rlen': L})
    region, bed_start, vl, _ = H.dense_variant_region(3, alt_n=False)
    rid = e.load_region(region, bed_start)
    cp = e.build_copy(rid, vl)
    rs = np.random.RandomState(5)
    n = 4000
    ts = rs.randint(cp.p_min, cp.p_max - 2 * L, size=n).astype(np.int64)
    tl = rs.randint(L, 2 * L, size=n).astype(np.int64)
    fo = rs.randint(0, 2, size=n).astype(np.int8)
    te = ts + tl
    assert ((te < cp.p_max) & (ts >= cp.p_min)).all()                          # only the N filter drops templates
    sample, chrom = LONG_NAMES['max']
    o1, o2, ocnt = oracle.generate_unit(region, bed_start + 1, H.oracle_cv(vl), L, ts, te, fo, '{}:0:0'.format(sample), chrom, 0)
    assert ocnt > 0.8 * n
    out = (np.empty(len(o1) + 64, dtype=np.uint8), np.empty(len(o1) + 64, dtype=np.uint8))
    e.prof_reset()
    f1, f2, cnt, nk, nb = e.generate_unit(cp, n, 0.5, MODE_EXPLICIT, 0, '@{}:0:0:'.format(sample), '|{}|0'.format(chrom),
                                          ts=ts, tl=tl, fo=fo, out=out)
    assert e.prof()['emit_launches'] == 2
    assert (cnt, nk, nb) == (ocnt, n, len(o1))
    assert f1.tobytes() == o1 and f2.tobytes() == o2
    e.free_copy(cp); e.free_region(rid)
  finally:
    e.close()


# ---- 6. k_unit_plan's tile protocol ------------------------------------------------------------------

PLAN_L = 12
PLAN_COUNTS = [1, 255, 256, 257, 31 * 256 + 1, 32 * 256, 32 * 256 + 1, 128 * 256, 128 * 256 + 1, 129 * 256 + 3, 1000 * 256 + 5]
EMPTY_RUNS = [1, 31, 32, 127, 128, 129, 300]
PLAN_BED = 1000                 # BED start of the plan tests' region: a template start below p_min stays positive
N_RUN = (150000, 210000)        # region offsets of its N run


@pytest.fixture(scope='module')
def plan_contig():
  seq = synth.synth_contig(400000, seed=17)
  seq[N_RUN[0]:N_RUN[1]] = ord('N')
  return seq


def tile_kinds(n_tiles, pattern):
  """Per tile: 'K' kept (in the run patterns with a few candidates dropped), 'T' nothing passes the te
  test, 'N' everything passes it and fails the N filter."""
  if pattern == 'all':
    return ['K'] * n_tiles
  if pattern == 'none':
    return ['T'] * n_tiles
  empty = 'T' if pattern == 'te_runs' else 'N'
  kinds = []
  for r in EMPTY_RUNS:
    kinds += ['K'] + [empty] * r
  kinds += ['K'] * max(0, n_tiles - len(kinds))
  return kinds[:n_tiles]


def plan_templates(n, pattern, p_min, p_max, rs):
  """Explicit (ts, tl, fo) for n candidates laid out tile by tile after tile_kinds."""
  L = PLAN_L
  kinds = np.repeat(np.array(tile_kinds((n + PLAN_TILE - 1) // PLAN_TILE, pattern)), PLAN_TILE)[:n]
  if pattern in ('te_runs', 'n_runs'):                     # kept tiles lose a random quarter, to either filter
    drop = (kinds == 'K') & (rs.rand(n) < 0.25)
    kinds[drop] = np.where(rs.rand(drop.sum()) < 0.5, 'T', 'N')
  clean = p_min + np.concatenate([np.arange(0, N_RUN[0] - 100), np.arange(N_RUN[1] + 1, p_max - p_min - 100)])
  ts = clean[rs.randint(0, clean.size, size=n)].astype(np.int64)
  tl = rs.randint(0, 4 * L, size=n).astype(np.int64)
  t = kinds == 'T'
  low = t & (rs.rand(n) < 0.5)                              # ts < p_min, or te >= p_max
  ts[low] = p_min - 1 - rs.randint(0, 5, size=low.sum())
  ts[t & ~low] = p_max - L + rs.randint(0, 5, size=(t & ~low).sum())
  nn = kinds == 'N'
  ts[nn] = p_min + rs.randint(N_RUN[0], N_RUN[1] - 100, size=nn.sum())    # read 1 lies in the N run
  fo = rs.randint(0, 2, size=n).astype(np.int8)
  return ts, tl, fo


def plan_unit(eng, cp, ref, n, pattern, seed):
  """One explicit unit: n_te_kept == numpy, count and bytes == oracle, serials 1..cnt.  -> file 1."""
  from mitty_b200.engine import MODE_EXPLICIT
  rs = np.random.RandomState(seed)
  ts, tl, fo = plan_templates(n, pattern, cp.p_min, cp.p_max, rs)
  f1, f2, cnt, nk, nb = eng.generate_unit(cp, n, 0.5, MODE_EXPLICIT, 0, '@P:0:0:', '|p|0', ts=ts, tl=tl, fo=fo)
  te = ts + np.maximum(tl, PLAN_L)
  keep = (te < cp.p_max) & (ts >= cp.p_min)
  assert nk == keep.sum(), (n, pattern)
  o1, o2, ocnt = oracle.generate_unit(ref, PLAN_BED + 1, H.oracle_cv(vcfio.VariantList.from_variants([])), PLAN_L, ts[keep], te[keep], fo[:keep.sum()],
                                      'P:0:0', 'p', 0)
  assert cnt == ocnt, (n, pattern)
  assert f1.tobytes() == o1 and f2.tobytes() == o2, (n, pattern)
  if pattern == 'none':
    assert (cnt, nk, nb) == (0, 0, 0)
  elif pattern == 'n_runs' and n > PLAN_TILE:
    assert cnt < nk                                        # the N filter dropped what the te test kept
  serials = [int(h[len(b'@P:0:0:'):h.index(b'|')]) for h in o1.split(b'\n')[0::4][:-1]]
  assert serials == list(range(1, cnt + 1))
  return f1.tobytes()


@pytest.mark.parametrize('pattern', ['all', 'none', 'te_runs', 'n_runs'])
def test_plan_tile_edges(eng, plan_contig, pattern):
  """Candidate counts on the edges of a tile, of the 32-tile and 128-descriptor look-back windows and
  beyond the 888 resident CTAs of a B200 (CTAs take several tiles), with runs of 1 ... 300 tiles that keep
  nothing and tiles emptied by the N filter alone (the te-survivor and kept counts drift apart)."""
  eng.load_model({'cum_tlen': np.array([1.0]), 'cum_bq_mat': np.ones((2, 300, 94)), 'rlen': PLAN_L})
  rid = eng.load_region(plan_contig, PLAN_BED)
  cp = eng.build_copy(rid, vcfio.VariantList.from_variants([]))
  for n in PLAN_COUNTS:
    plan_unit(eng, cp, plan_contig, n, pattern, n)
  eng.free_copy(cp); eng.free_region(rid)


def test_plan_state_between_units(eng, plan_contig):
  """A large unit, a one-tile unit and the large unit again on one engine: identical bytes (nothing is
  left behind in the tile descriptors or the tile counter)."""
  eng.load_model({'cum_tlen': np.array([1.0]), 'cum_bq_mat': np.ones((2, 300, 94)), 'rlen': PLAN_L})
  rid = eng.load_region(plan_contig, PLAN_BED)
  cp = eng.build_copy(rid, vcfio.VariantList.from_variants([]))
  big = plan_unit(eng, cp, plan_contig, PLAN_COUNTS[-1], 'n_runs', 1)
  plan_unit(eng, cp, plan_contig, 200, 'all', 2)
  assert plan_unit(eng, cp, plan_contig, PLAN_COUNTS[-1], 'n_runs', 1) == big
  eng.free_copy(cp); eng.free_region(rid)


# ---- 7. standalone corrupt-reads in production mode ---------------------------------------------------

def fastq(names, seqs):
  return b''.join(b'@' + nm + b'\n' + sq + b'\n+\n' + b'#' * len(sq) + b'\n' for nm, sq in zip(names, seqs))


def corrupt_inputs(rs, giant=False):
  """Paired inputs: ragged lengths 1-5, 150, 299, 300 in every warp tile, lower-case and IUPAC letters,
  names of 0 ... 1000 bytes with and without comments (file 2 has names of its own).  giant: one name of
  13 KB, larger than the staged kernel's stage."""
  lens = [1, 2, 3, 4, 5, 150, 299, 300]
  name_lens = [0, 1, 3, 5, 300, 1000]
  n = 200
  names1, names2, s1, s2 = [], [], [], []
  letters = np.frombuffer(b'ACGTACGTACGTNacgtnRYKMSWBDHV', dtype=np.uint8)
  for k in range(n):
    nl = name_lens[k % len(name_lens)]
    nm = bytes(rs.choice(np.frombuffer(b'ABCxyz0189:_|/', dtype=np.uint8), size=nl))
    if (k // len(name_lens)) % 2:
      nm += [b' comment 1:N:0', b'\tx', b'\r'][k % 3]
    names1.append(nm)
    names2.append(b'mate2_' + str(k).encode() + b' other')
    for seqs in (s1, s2):
      L = lens[rs.randint(0, len(lens))]
      seqs.append(bytes(letters[rs.randint(0, letters.size, size=L)]))
  if giant:
    names1[37] = b'G' * 13000 + b' tail'
  return fastq(names1, s1), fastq(names2, s2)


@pytest.mark.parametrize('giant', [False, True])
@pytest.mark.parametrize('first', [0, 12345, (1 << 32) + 7])
def test_corrupt_reads_philox_exact(eng, giant, first):
  """eng.corrupt_fastq in production mode == the numpy specification (table 1, key 0x636f7232, serials
  from first_template, '@' + read 1's name on both files), paired and single-end.  With the 13 KB name the
  whole call goes to k_corrupt's Philox branch, so every other record of it is checked on that path."""
  from mitty_b200.engine import MODE_PHILOX
  m = H.model('hiseq-X-v2.5-Garvan.pkl')
  eng.load_model(m)
  tables = eng.model_tables(1)
  b1, b2 = corrupt_inputs(np.random.RandomState(3 + int(giant)), giant)
  big = max(2 * max(len(a), len(b)) + len(PR.record_name(h)) + 6
            for h, a, b in zip(b1.split(b'\n')[0::4], b1.split(b'\n')[1::4], b2.split(b'\n')[1::4]))
  assert (big + 16 > 32 * (2 * 150 + 6 + 96)) == giant      # MG_CORRUPT_STAGE: the staged kernel's limit
  n = b1.count(b'\n') // 4
  serials = np.arange(n, dtype=np.uint64) + np.uint64(first)
  cseed = 2024
  c1, c2, cnt = eng.corrupt_fastq(b1, b2, mode=MODE_PHILOX, seed=cseed, first_template=first)
  assert cnt == n
  assert c1.tobytes() == PR.corrupt_file(b1, 0, tables, cseed, CORRUPT_KEY, serials=serials, names_from=b1)
  assert c2.tobytes() == PR.corrupt_file(b2, 1, tables, cseed, CORRUPT_KEY, serials=serials, names_from=b1)
  s1, s2, scnt = eng.corrupt_fastq(b1, None, mode=MODE_PHILOX, seed=cseed, first_template=first)
  assert scnt == n and s2 is None
  assert s1.tobytes() == c1.tobytes()
  if not giant:   # long names split the staged kernel's batches (k_corrupt_staged batches a warp tile as k_unit_emit does)
    tiles = stage_batches(*record_bounds(c1.tobytes()), 32 * (2 * 150 + 6 + 96) & ~15)
    assert np.mean([len(t) > 1 for t in tiles]) > 0.5
