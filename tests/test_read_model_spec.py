"""bam2illumina without a device: the model derivation against the five shipped models, the specification
(tests/read_model_spec.py) against hand-computed counts, the .pkl writer, and the native BGZF BAM reader
(mg_bam_scan) on chosen member layouts and malformed files."""
import glob
import os
import pickle
import struct

import numpy as np
import pytest

from tests import read_model_spec as S

MODELS = sorted(glob.glob(os.path.join(os.path.dirname(__file__), '..', 'mitty_b200', 'data', 'readmodels', '*.npz')))


@pytest.mark.parametrize('path', MODELS, ids=[os.path.basename(p)[:-4] for p in MODELS])
def test_derivation_reproduces_shipped_models(path):
  from mitty_b200.empirical.bam2illumina import model_from_counts
  z = np.load(path)
  bq, tlen = z['bq_mat'], z['tlen']
  per_cycle = np.append(bq.sum(axis=(0, 2)), np.uint64(0))
  len_hist = np.zeros(bq.shape[1] + 1, dtype=np.uint64)
  len_hist[1:] = per_cycle[:-1] - per_cycle[1:]           # reads of length L: cycle L-1 counted, cycle L not
  m = model_from_counts(bq, len_hist, tlen, 'x')
  for k in ('cum_bq_mat', 'cum_tlen'):
    assert m[k].dtype == np.float64 and m[k].tobytes() == z[k].tobytes(), k
  for k in ('r_cnt', 'min_rlen', 'max_rlen', 'mean_rlen'):
    assert m[k] == int(z[k]) and type(m[k]) is int, k
  assert m['model_class'] == 'illumina' and m['bq_mat'].dtype == np.uint64 and m['tlen'].dtype == np.uint64


def test_mean_rlen_is_the_mode_ties_to_the_longer():
  from mitty_b200.empirical.bam2illumina import model_from_counts
  bq = np.zeros((2, 10, 94), dtype=np.uint64)
  lh = np.zeros(11, dtype=np.uint64)
  lh[[3, 7, 9]] = [5, 5, 2]
  m = model_from_counts(bq, lh, np.ones(4, dtype=np.uint64), 'x')
  assert (m['min_rlen'], m['max_rlen'], m['mean_rlen']) == (3, 9, 7)
  assert not m['cum_bq_mat'].any()
  with pytest.raises(ValueError, match='no read'):
    model_from_counts(bq, np.zeros(11, dtype=np.uint64), np.ones(4, dtype=np.uint64), 'x')


def _rules_records():
  """Records hitting every rule, with their expected effect computed by hand below."""
  R = S.record
  return [
    R(flag=0x41, seq=b'ACGT', qual=[10, 20, 30, 40], tlen=250),                      # 0 mate 0 forward, tlen 250
    R(flag=0x91, seq=b'ACG', qual=[5, 6, 99], tlen=-250),                            # 1 mate 1 reverse, q 99 -> 93
    R(flag=0x4, seq=b'AC', qual=[1, 1]),                                             # 2 unmapped
    R(flag=0x100, seq=b'AC', qual=[1, 1]),                                           # 3 secondary
    R(flag=0x200, seq=b'AC', qual=[1, 1]),                                           # 4 QC fail
    R(flag=0x800, seq=b'AC', qual=[1, 1]),                                           # 5 supplementary
    R(flag=0x400, seq=b'A', qual=[7]),                                               # 6 duplicate: counted, unpaired -> mate 0
    R(flag=0x41, mapq=10, seq=b'AC', qual=[1, 1], tlen=5),                           # 7 mapq 10
    R(flag=0x41, seq=b'', qual=[], tlen=5),                                          # 8 empty SEQ
    R(flag=0x41, seq=b'AC', qual=None, tlen=5),                                      # 9 missing QUAL
    R(flag=0x41, seq=b'A' * 6, qual=[2] * 6, tlen=5),                                # 10 longer than max_bp = 5
    R(flag=0x41, seq=b'AC', qual=[3, 4], tlen=-2 ** 31),                             # 11 INT32_MIN: |TLEN| = 2^31, not counted
    R(flag=0x51, seq=b'ACGTA', qual=[0, 1, 2, 3, 4], tlen=1000, cigar=((3, 5), (5, 0))),  # 12 reverse mate 0, hard clip, tlen >= max_tlen
    R(flag=0x81, seq=b'AC', qual=[8, 9], tlen=-3),                                   # 13 mate 1 forward: its TLEN is not counted
  ]


def test_spec_rules_hand_computed():
  recs = _rules_records()
  c = S.count_records(recs, max_bp=5, max_tlen=1000, min_mq=20)
  bq = np.zeros((2, 5, 94), dtype=np.uint64)
  for mate, cyc, q in ((0, 0, 10), (0, 1, 20), (0, 2, 30), (0, 3, 40),     # 0
                       (1, 0, 93), (1, 1, 6), (1, 2, 5),                    # 1 reversed
                       (0, 0, 7),                                           # 6
                       (0, 0, 3), (0, 1, 4),                                # 11
                       (0, 0, 4), (0, 1, 3), (0, 2, 2), (0, 3, 1), (0, 4, 0),  # 12 reversed
                       (1, 0, 8), (1, 1, 9)):                               # 13
    bq[mate, cyc, q] += 1
  assert np.array_equal(c['bq_mat'], bq)
  lh = np.zeros(6, dtype=np.uint64)
  lh[[4, 3, 1, 2, 5]] = [1, 1, 1, 2, 1]
  lh[2] = 2
  assert np.array_equal(c['len_hist'], lh)
  tl = np.zeros(1000, dtype=np.uint64)
  tl[250] = 1                                  # record 0 only: 1 is mate 1, 11 and 12 are beyond max_tlen
  assert np.array_equal(c['tlen'], tl)
  assert (c['records'], c['considered'], c['counted']) == (14, 14, 6)
  assert [c[k] for k in S.SKIPS] == [4, 1, 1, 1, 1]
  e = S.count_records(recs, max_bp=5, every=3)                 # ordinals 0, 3, 6, 9, 12
  assert (e['considered'], e['counted'], e['skip_flag'], e['skip_noqual']) == (5, 3, 1, 1)


def test_pkl_round_trip(tmp_path):
  from click.testing import CliRunner
  from mitty_b200.cli import cli
  from mitty_b200.empirical.bam2illumina import model_from_counts, write_model
  from mitty_b200.readmodels import get_read_model, load_model
  z = np.load(MODELS[0])
  m = model_from_counts(z['bq_mat'], np.bincount([100, 100, 150], minlength=301).astype(np.uint64), z['tlen'], 'my sequencer', min_mq=20)
  d = tmp_path / 'models'
  d.mkdir()
  pkl = str(d / 'mine.pkl')
  umask = os.umask(0o022)
  try:
    write_model(pkl, m)
  finally:
    os.umask(umask)
  assert os.listdir(str(d)) == ['mine.pkl']
  assert os.stat(pkl).st_mode & 0o777 == 0o644                  # as open() would create it, not mkstemp's 0600
  back = load_model(pkl)
  assert sorted(back) == sorted(m)
  for k, v in m.items():
    assert type(back[k]) is type(v) and (np.array_equal(back[k], v) if isinstance(v, np.ndarray) else back[k] == v), k
  module, model = get_read_model(pkl)
  assert module.__name__.endswith('illumina') and model['mean_rlen'] == 100
  res = CliRunner().invoke(cli, ['list-read-models', '-d', str(d)])
  assert res.exit_code == 0 and 'mine.pkl' in res.output and 'my sequencer' in res.output


# ---- the native reader without a device -----------------------------------------------------------------

def _raw(n=600, seed=3, contigs=(('c', 100000), ('d', 5000))):
  rng = np.random.RandomState(seed)
  recs = []
  for k in range(n):
    l = int(rng.randint(0, 160))
    recs.append(S.record(name=b'read%d' % k, flag=int(rng.choice([0x41, 0x81, 0x51, 0x91, 0, 0x10, 0x4])), mapq=int(rng.randint(0, 61)),
                         seq=bytes(rng.choice(list(b'ACGTN'), l).tolist()), qual=[int(x) for x in rng.randint(2, 42, l)], tlen=int(rng.randint(-900, 900)),
                         tags=b'RGZx\0' * int(rng.randint(0, 3))))
  return S.header(contigs, text='@HD\tVN:1.4\n' + '@CO\t' + 'x' * 3000 + '\n') + b''.join(recs), n


def _scan(path, **kw):
  from mitty_b200.engine import scan_bam
  return scan_bam(path, **kw)


LAYOUTS = {
  'fixed': dict(cuts=65280),
  'small_members': dict(cuts=997),
  'one_byte_and_empty': dict(cuts=[1, 1, 1, 37, 1, 4096, 1, 2], empty_every=2),
  'level0': dict(cuts=5000, level=0),
  'mixed_levels': dict(cuts=3000, level=lambda k: (0, 1, 9)[k % 3]),
  'extra_subfields': dict(cuts=20000, extra=b'XY\x03\x00abc' + b'ZZ\x00\x00'),
}


@pytest.mark.parametrize('layout', sorted(LAYOUTS))
@pytest.mark.parametrize('threads,chunk', [(1, 1 << 17), (3, 1 << 20), (16, 64 << 20)])
def test_reader_layouts(tmp_path, layout, threads, chunk):
  raw, n = _raw()
  data = S.bgzf(raw, **LAYOUTS[layout])
  assert b''.join(r for _, r in S.members(data)) == raw
  p = str(tmp_path / 'x.bam')
  open(p, 'wb').write(data)
  got = _scan(p, threads=threads, chunk_bytes=chunk)
  assert got == {'records': n, 'inflated_bytes': len(raw), 'compressed_bytes': len(data), 'eof_marker': 1}


def test_reader_fname_member_and_large_record(tmp_path):
  """A member with FNAME, and a record longer than the chunk buffer (it grows)."""
  big = S.record(seq=b'A' * 400000, qual=[30] * 400000)
  raw = S.header() + S.record() + big + S.record()
  data = S.member(raw[:50], fname=b'name.bam') + S.bgzf(raw[50:], cuts=60000)
  p = str(tmp_path / 'x.bam')
  open(p, 'wb').write(data)
  assert _scan(p, threads=2, chunk_bytes=1 << 17)['records'] == 3


def test_reader_missing_eof_marker(tmp_path):
  raw, n = _raw(50)
  p = str(tmp_path / 'x.bam')
  open(p, 'wb').write(S.bgzf(raw, cuts=4000, eof=False))
  assert _scan(p) == {'records': n, 'inflated_bytes': len(raw), 'compressed_bytes': len(S.bgzf(raw, cuts=4000, eof=False)), 'eof_marker': 0}


def _tampered(case):
  """-> (BGZF bytes, expected ('offset' | 'record', where)) of one malformed input."""
  raw, n = _raw(200)
  cut = 7000
  data = S.bgzf(raw, cuts=cut)
  offs = [o for o, _ in S.members(data)]
  recs = S.records(raw)
  start = len(raw) - sum(len(r) for r in recs)           # first record's offset in the stream
  at = [start + sum(len(r) for r in recs[:k]) for k in range(len(recs) + 1)]
  if case == 'not_gzip':
    b = bytearray(data); b[offs[3]] = 0x1e
    return bytes(b), ('offset', offs[3])
  if case == 'no_bc':
    b = bytearray(data); b[offs[2] + 12] = ord('X')
    return bytes(b), ('offset', offs[2])
  if case == 'crc':
    b = bytearray(data); b[offs[4 + 1] - 8] ^= 1
    return bytes(b), ('offset', offs[4])
  if case == 'isize':
    b = bytearray(data); b[offs[5 + 1] - 4] ^= 1
    return bytes(b), ('offset', offs[5])
  if case == 'corrupt_deflate':
    b = bytearray(data); b[offs[1] + 20] ^= 0xFF; b[offs[1] + 21] ^= 0xFF
    return bytes(b), ('offset', offs[1])
  if case == 'truncated_member':
    return data[:offs[3] + 100], ('offset', offs[3])
  if case == 'magic':
    return S.bgzf(b'BAM\x02' + raw[4:], cuts=cut), ('offset', 0)
  if case == 'block_size':
    k = 77
    r = bytearray(raw); r[at[k]:at[k] + 4] = struct.pack('<i', 31)
    return S.bgzf(bytes(r), cuts=cut), ('record', k)
  if case == 'cut_record':
    return S.bgzf(raw[:at[150] + 40], cuts=cut), ('record', 150)
  raise KeyError(case)


FRAMING = ['not_gzip', 'no_bc', 'crc', 'isize', 'corrupt_deflate', 'truncated_member', 'magic', 'block_size', 'cut_record']


@pytest.mark.parametrize('case', FRAMING)
def test_spec_and_reader_reject_malformed(tmp_path, case):
  data, (kind, where) = _tampered(case)
  with pytest.raises(S.SpecError) as e:
    S.counts(data)
  assert (e.value.kind, e.value.where) == (kind, where)
  p = str(tmp_path / 'bad.bam')
  open(p, 'wb').write(data)
  for threads, chunk in ((1, 1 << 17), (4, 1 << 22)):
    with pytest.raises(ValueError, match='{} {}:'.format('record' if kind == 'record' else 'compressed offset', where)):
      _scan(p, threads=threads, chunk_bytes=chunk)


def test_reader_header_errors(tmp_path):
  p = str(tmp_path / 'h.bam')
  open(p, 'wb').write(S.bgzf(S.header()[:20]))
  with pytest.raises(ValueError, match='ends inside the BAM header'):
    _scan(p)
  open(p, 'wb').write(b'')
  with pytest.raises(ValueError, match='ends inside the BAM header'):
    _scan(p)
  open(p, 'wb').write(b'plain text, not BGZF at all')
  with pytest.raises(ValueError, match='compressed offset 0: not a gzip member'):
    _scan(p)
  raw = S.header() + S.record()
  open(p, 'wb').write(pickle.dumps(raw))
  with pytest.raises(ValueError, match='compressed offset 0'):
    _scan(p)
