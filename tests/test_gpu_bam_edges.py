"""god-aligner on the device at the shapes real genomes give it, byte for byte against the pure-Python
specification (tests/bam_spec.py): the decompressed BAM equals ``S.bam_bytes`` and the index equals
``S.build_bai``.

- k_radix_hist / k_radix_scatter: 1 to 6 passes of 8 bits (GRCh37, hs37d5-like and GRCh38-with-alts-shaped
  contig tables), tiles of 4096 keys at and around their edges, ties across tiles;
- reg2bin and the index at every level of the binning scheme, up to a contig of exactly 2^29 bases;
- the merge of spilled runs (key and record buffers refilled, a record larger than the record buffer) and the
  writer's path for a record that straddles two device-to-host pieces;
- record-level edges (name lengths, odd lengths on strand 1, every nt16 letter, every quality, mates at one
  position, a mate inside an insertion);
- contigs BAM cannot address (2^31 bases or more: rejected) or BAI cannot index (past 2^29: no index, the
  bin's low 16 bits).

The engine's BamWriter is driven directly with a declared contig table, so a test can declare a 2^29-base
contig or 3 366 contigs without writing a FASTA.  Every test restates the host rule it targets and asserts
that its inputs reach the path it is named after."""
import logging
import math
import os
import random
import struct

import numpy as np
import pytest

from tests import bam_spec as S

pytestmark = pytest.mark.gpu

# host rules of mg_bam.cu, restated
DIGIT_BITS = 8            # sort_run: passes = max(1, ceil(key_bits / 8))
RADIX_TILE = 4096         # RS_TILE: keys per tile of k_radix_hist / k_radix_scatter
PER_READ = 72             # kPerRead: a run fits while 2 * record bytes + 72 * reads <= run_bytes
MERGE_KEYS = 1 << 16      # RunReader: keys read 65 536 at a time ...
MERGE_RECORDS = 4 << 20   # ... and records through a 4 MiB buffer that grows for a larger record
PIECE = 64 << 20          # kPiece: one run goes device-to-host in 64 MB pieces


@pytest.fixture(scope='module')
def eng():
  from mitty_b200.engine import Engine
  e = Engine(0)
  yield e
  e.close()


def key_bits(contigs):
  """mg_bam_open: key = refID << (pos_bits + 1) | pos << 1 | reverse, pos_bits = bit_length(longest contig)."""
  return (len(contigs) - 1).bit_length() + max(1, max(l for _, l in contigs)).bit_length() + 1


def passes(contigs):
  return max(1, -(-key_bits(contigs) // DIGIT_BITS))


def record_keys(contigs, recs):
  """The sort key of each encoded record (refID, POS, FLAG 0x10), as the device forms it."""
  pb = max(1, max(l for _, l in contigs)).bit_length()
  out = []
  for r in recs:
    ref, pos, fnc = struct.unpack_from('<iiI', r, 4)[0], struct.unpack_from('<i', r, 8)[0], struct.unpack_from('<I', r, 16)[0]
    out.append(ref << (pb + 1) | pos << 1 | (fnc >> 20 & 1))
  return out


def write(eng, path, contigs, chunks, bai=True, run_bytes=None, level=1, threads=4):
  """BamWriter over FASTQ chunks [(fq1, fq2 or None)]: add until each chunk is consumed, then close, as
  god_aligner.process_multi_threaded does.  -> (records, runs)"""
  from mitty_b200.engine import BamWriter
  bw = BamWriter(eng, path, path + '.bai' if bai else None, contigs, S.header_text(contigs, 'S'), 'S', level=level, threads=threads,
                 run_bytes=run_bytes)
  try:
    for fq1, fq2 in chunks:
      a1 = np.frombuffer(fq1, np.uint8)
      a2 = np.frombuffer(fq2, np.uint8) if fq2 is not None else None
      while a1.size:
        n, c1, c2 = bw.add(a1, a2)
        assert n > 0
        a1 = a1[c1:]
        a2 = a2[c2:] if a2 is not None else None
    n, runs, _ = bw.close()
  finally:
    bw.abort()
  return n, runs


def check(path, contigs, fq1, fq2=None, bai=True, recs=None):
  """The BAM (and index) equal the specification (``recs``: the spec's records, when already built).
  -> (file bytes, the spec's sorted records)"""
  data = open(path, 'rb').read()
  sample, recs = S.records(contigs, fq1, fq2) if recs is None else ('S', recs)
  assert S.decompress(data) == S.header_bytes(contigs, sample) + b''.join(recs)
  if bai:
    assert open(path + '.bai', 'rb').read() == S.build_bai(data, len(contigs))
  else:
    assert not os.path.exists(path + '.bai')
  return data, recs


def seq_of(rng, n, letters=b'ACGT'):
  return bytes(rng.choice(letters) for _ in range(n))


def read(rng, pos0, span, strand=None):
  pos, cig, rlen = S.read_layout(pos0, span)
  return (rng.randrange(2) if strand is None else strand, pos, cig, seq_of(rng, rlen), bytes(rng.randrange(35, 75) for _ in range(rlen)))


# ---- 1. radix pass counts -----------------------------------------------------------------------------

GRCH37 = [('1', 249250621), ('2', 243199373), ('3', 198022430), ('4', 191154276), ('5', 180915260), ('6', 171115067), ('7', 159138663),
          ('8', 146364022), ('9', 141213431), ('10', 135534747), ('11', 135006516), ('12', 133851895), ('13', 115169878), ('14', 107349540),
          ('15', 102531392), ('16', 90354753), ('17', 81195210), ('18', 78077248), ('19', 59128983), ('20', 63025520), ('21', 48129895),
          ('22', 51304566), ('X', 155270560), ('Y', 59373566), ('MT', 16569)]
GRCH38 = [('chr' + n if n != 'MT' else 'chrM', l) for n, l in
          [('1', 248956422), ('2', 242193529), ('3', 198295559), ('4', 190214555), ('5', 181538259), ('6', 170805979), ('7', 159345973),
           ('8', 145138636), ('9', 138394717), ('10', 133797422), ('11', 135086622), ('12', 133275309), ('13', 114364328), ('14', 107043718),
           ('15', 101991189), ('16', 90338345), ('17', 83257441), ('18', 80373285), ('19', 58617616), ('20', 64444167), ('21', 46709983),
           ('22', 50818468), ('X', 156040895), ('Y', 57227415), ('MT', 16569)]]


def grch38_with_alts():
  """3 366 contigs named as GRCh38's analysis set with alts, decoys and HLA alleles (lengths made up)."""
  rng = random.Random(38)
  out = list(GRCH38)
  k = 0
  while len(out) < 3366:
    c = GRCH38[k % 24][0]
    kind = k % 5
    name = ('{}_KI{}v1_alt'.format(c, 270700 + k) if kind == 0 else '{}_GL{}v1_random'.format(c, 383500 + k) if kind == 1 else
            'chrUn_JTFH0100{:04d}v1_decoy'.format(k) if kind == 2 else 'HLA-{}*{:02d}:{:02d}:01:{:02d}'.format('ABC'[k % 3], k % 97, k % 89, k % 7)
            if kind == 3 else 'chrEBV_{}'.format(k))
    out.append((name, rng.randrange(1000, 400000)))
    k += 1
  return out


GENOMES = {
    8: [('chrM', 100)],
    9: [('chrM', 100), ('phiX', 120)],
    16: [('a', 5000), ('b', 8000), ('c', 6000)],
    17: [('a', 5000), ('b', 8000), ('c', 6000), ('d', 100), ('e', 7000)],
    28: [('chr1', 50000000), ('chr2', 48000000)],
    32: [('chr%d' % (i + 1), 40000000 - 1500000 * i) for i in range(20)],
    34: GRCH37,
    41: None,
}


def log_uniform_templates(rng, contigs, n, L=30):
  """Paired templates at log-uniform positions up to each contig's last base, on the first, the last and
  random contigs, both strands; a template ends on the last base of the first and of the last contig."""
  out = []
  for t in range(n):
    ref = 0 if t % 7 == 0 else len(contigs) - 1 if t % 7 == 1 else rng.randrange(len(contigs))
    chrom, length = contigs[ref]
    rl = min(L, length)
    reads = []
    for _ in range(2):
      pos0 = min(length - rl, int(math.exp(rng.uniform(0, math.log(length)))) - 1)
      reads.append((rng.randrange(2), pos0 + 1, '%d=' % rl, seq_of(rng, rl), b'F' * rl))
    out.append((chrom, reads))
  for ref in (0, len(contigs) - 1):
    chrom, length = contigs[ref]
    rl = min(L, length)
    out.append((chrom, [(1, length - rl + 1, '%d=' % rl, seq_of(rng, rl), b'F' * rl)] * 2))
  return out


@pytest.mark.parametrize('bits', sorted(GENOMES))
def test_radix_pass_counts(tmp_path, eng, bits):
  contigs = GENOMES[bits] or grch38_with_alts()
  assert key_bits(contigs) == bits
  n_pass = passes(contigs)
  rng = random.Random(bits)
  fq1, fq2 = S.fastq(log_uniform_templates(rng, contigs, 3000))
  p = str(tmp_path / 'p.bam')
  assert write(eng, p, contigs, [(fq1, fq2)]) == (6004, 1)
  _, recs = check(p, contigs, fq1, fq2)
  # guard: each pass's digit takes several values among the keys, and the top pass's digit is not always 0
  keys = record_keys(contigs, recs)
  for d in range(n_pass):
    digits = {k >> (DIGIT_BITS * d) & 255 for k in keys}
    assert len(digits) >= min(3, 1 << (bits - DIGIT_BITS * d)), (d, sorted(digits))
  assert any(k >> (DIGIT_BITS * (n_pass - 1)) for k in keys)


def test_radix_pass_counts_cover_one_to_six():
  """The contig tables above give 1 - 6 passes: a single pass, even counts (the sorted keys copied back into
  d_key2 / d_ord2) and digit shifts of 24 bits and more."""
  got = sorted({passes(c or grch38_with_alts()) for c in GENOMES.values()})
  assert got == [1, 2, 3, 4, 5, 6]


# ---- 2. tiles and stability -----------------------------------------------------------------------------

COUNTS = [1, 2, 255, 256, 4095, 4096, 4097, 3 * 4096 + 17]
TILE_CONTIGS = [('t', 1 << 17), ('u', 1000)]


def pattern_templates(rng, pattern, n, paired):
  """n templates whose records (template by template, file 1 first) have keys all equal, strictly
  descending, from three values, or random with many duplicates."""
  nf = 2 if paired else 1
  R = n * nf
  if pattern == 'three':
    trio = [(500, 0), (500, 1), (70000, 0)]
  out = []
  for t in range(n):
    reads = []
    for f in range(nf):
      r = t * nf + f
      if pattern == 'equal':
        pos0, strand = 1000, 0
      elif pattern == 'descending':
        pos0, strand = (R - r) >> 1, (R - r) & 1
      elif pattern == 'three':
        pos0, strand = trio[rng.randrange(3)]
      else:
        pos0, strand = rng.randrange(max(1, R // 16)), rng.randrange(2)
      reads.append((strand, pos0 + 1, '3=', seq_of(rng, 3), b'III'))
    out.append(('t', reads))
  return out


@pytest.mark.parametrize('paired', [False, True], ids=['single', 'paired'])
@pytest.mark.parametrize('pattern', ['equal', 'descending', 'three', 'duplicates'])
def test_radix_tiles_and_stability(tmp_path, eng, pattern, paired):
  rng = random.Random(pattern)
  tiles_seen = set()
  for n in COUNTS:
    fq1, fq2 = S.fastq(pattern_templates(rng, pattern, n, paired))
    p = str(tmp_path / ('t%d.bam' % n))
    R = n * (2 if paired else 1)
    assert write(eng, p, TILE_CONTIGS, [(fq1, fq2)]) == (R, 1)
    _, recs = check(p, TILE_CONTIGS, fq1, fq2)
    # guard: tile count and fill of the last tile; ties that span tiles where the pattern has ties
    tiles_seen.add((-(-R // RADIX_TILE), R % RADIX_TILE))
    names = [r[36:36 + r[12] - 1] for r in recs]
    keys = record_keys(TILE_CONTIGS, recs)
    if R > RADIX_TILE and pattern != 'descending':
      order = {}
      for k, nm in zip(keys, names):
        order.setdefault(k, []).append(int(nm.split(b'|')[0].rsplit(b':', 1)[1]))
      assert any(v[0] < RADIX_TILE // (2 if paired else 1) <= v[-1] for v in order.values())
    if pattern == 'descending':
      assert len(set(keys)) == R
  assert {t for t, _ in tiles_seen} >= ({1, 2, 3} if paired else {1, 2, 4})
  assert any(f == 0 for _, f in tiles_seen) and any(0 < f < 32 for _, f in tiles_seen)


# ---- 3. bins and the index at every level ------------------------------------------------------------------

BIN_CONTIGS = [('chrA', 1 << 29), ('gap1', 5000), ('chrB', 3 * (1 << 26) + 12345), ('gap2', 7000), ('chrC', (1 << 20) + 7)]


def rec_span(r):
  """Reference length of an encoded record's CIGAR."""
  n = struct.unpack_from('<I', r, 16)[0] & 0xFFFF
  return sum(c >> 4 for c in struct.unpack_from('<%dI' % n, r, 36 + r[12]) if c & 15 in (0, 2, 3, 7, 8))


def level(b):
  return 0 if b == 0 else 1 if b < 9 else 2 if b < 73 else 3 if b < 585 else 4 if b < 4681 else 5


@pytest.mark.parametrize('layout', ['spread', 'one_contig'])
def test_bins_and_index_at_every_level(tmp_path, eng, layout):
  rng = random.Random(layout)
  refs = (0, 2, 4) if layout == 'spread' else (0, )
  templates = []
  for ref in refs:
    chrom, length = BIN_CONTIGS[ref]
    edges = S.bin_edge_spans(length)
    rng.shuffle(edges)
    # mates: two alignments at bin edges of one contig
    templates += [(chrom, [read(rng, *edges[i]), read(rng, *edges[i - 1])]) for i in range(len(edges))]
  fq1, fq2 = S.fastq(templates)
  p = str(tmp_path / 'b.bam')
  assert write(eng, p, BIN_CONTIGS, [(fq1, fq2)])[0] == 2 * len(templates)
  data, recs = check(p, BIN_CONTIGS, fq1, fq2)
  # guard: records in all six levels of the binning scheme, zero-span reads, a read ending on the 2^29th base
  bins = [struct.unpack_from('<H', r, 14)[0] for r in recs]
  assert {level(b) for b in bins} == set(range(6))
  ends = [(struct.unpack_from('<i', r, 4)[0], struct.unpack_from('<i', r, 8)[0] + rec_span(r)) for r in recs]
  assert (0, 1 << 29) in ends
  assert any(rec_span(r) == 0 for r in recs)
  regions = [q for ref in refs for q in S.edge_queries(ref, BIN_CONTIGS[ref][1])] + [(1, 0, 5000), (3, 0, 7000)]
  S.check_queries(data, open(p + '.bai', 'rb').read(), regions)


# ---- 4. merge and writer buffers ---------------------------------------------------------------------------

MERGE_CONTIGS = [('m', 1000000)]


def long_name_fastq(blocks, L=20):
  """Single-end FASTQ of the blocks' (strand, pos, cigar) reads, L bases each, names of exactly 254 bytes."""
  rng = random.Random(3)
  templates = [('m', [(s, p, c, seq_of(rng, L), b'A' * L)]) for b in blocks for s, p, c in b]
  fq1, _ = S.fastq(templates)
  pad = [255 - len(line) for line in fq1.split(b'\n')[0:-1:4]]   # '@' + 254 bytes
  return S.fastq(templates, pad=pad)[0]


def test_merge_of_large_runs_and_pieces(tmp_path, eng):
  B = MERGE_KEYS + 4464                                            # 70 000 records a run
  rng = random.Random(5)
  keys = [(rng.randrange(2), rng.randrange(1, 30000)) for _ in range(B)]
  # the same keys in every run; spans of 20 and 16 385 bases put the records of one key from consecutive runs
  # in different bins, so index chunks are short and the record that straddles a piece edge can begin or end one
  cigars = ['10=1X9=', '10=16365D10=', '10=1X9=']
  fq = long_name_fastq([[(s, p, c) for s, p in keys] for c in cigars])
  lines = fq.split(b'\n')
  cut = [b'\n'.join(lines[4 * B * j:4 * B * (j + 1)]) + b'\n' for j in range(3)]
  assert b''.join(cut) == fq
  _, recs = S.records(MERGE_CONTIGS, fq)
  assert {r[12] for r in recs} == {255}
  run_rec = [0, 0, 0]
  for r in recs:
    run_rec[int(r[36:36 + 254].split(b'|')[0].rsplit(b':', 1)[1]) // B] += len(r)
  run_bytes = 2 * run_rec[0] + PER_READ * B                        # one chunk fills a run exactly
  # guard: every spilled run refills the merge's key buffer and its record buffer, every key is in every run
  # (ties go to the earlier run); the single run is longer than a piece and a record straddles a piece edge
  assert B > MERGE_KEYS and min(run_rec) > MERGE_RECORDS and len(set(run_rec)) == 1
  assert len(set(keys)) > 10000
  rec_starts = np.cumsum([0] + [len(r) for r in recs])
  j = int(np.searchsorted(rec_starts, PIECE, side='right')) - 1
  bins = [struct.unpack_from('<H', r, 14)[0] for r in recs[j - 1:j + 2]]
  # ... and it begins or ends an index chunk, so its offsets reach the index
  assert rec_starts[-1] > PIECE and rec_starts[j] < PIECE and (bins[0] != bins[1] or bins[1] != bins[2])
  one = str(tmp_path / 'one.bam')
  assert write(eng, one, MERGE_CONTIGS, [(fq, None)], threads=8) == (3 * B, 1)
  check(one, MERGE_CONTIGS, fq, recs=recs)
  many = str(tmp_path / 'many.bam')
  assert write(eng, many, MERGE_CONTIGS, [(c, None) for c in cut], run_bytes=run_bytes, threads=8) == (3 * B, 3)
  assert open(many, 'rb').read() == open(one, 'rb').read() and open(many + '.bai', 'rb').read() == open(one + '.bai', 'rb').read()
  assert sorted(os.listdir(str(tmp_path))) == ['many.bam', 'many.bam.bai', 'one.bam', 'one.bam.bai']


def test_merge_of_a_record_larger_than_the_record_buffer(tmp_path, eng):
  rng = random.Random(7)
  rs = np.random.RandomState(7)
  contigs = [('big', 6000000), ('small', 50000)]
  L = 4600000
  big = ('big', [(1, 1000001, '%d=' % L, rs.choice(np.frombuffer(b'ACGTNacgt', np.uint8), L).tobytes(),
                  rs.randint(35, 75, L).astype(np.uint8).tobytes())])
  small = [('big', [read(rng, rng.randrange(0, 5990000), 100)]) for _ in range(1000)]
  chunks = [S.fastq(small[:500]), S.fastq([big]), S.fastq(small[500:])]
  big_rec = len(S.records(contigs, chunks[1][0])[1][0])
  # guard: the record outgrows the merge's 4 MiB record buffer; one such template alone fits a run, so the
  # runs are [500 small], [the big one], [500 small]
  assert big_rec > MERGE_RECORDS
  run_bytes = 2 * big_rec + PER_READ
  p = str(tmp_path / 'big.bam')
  assert write(eng, p, contigs, chunks, run_bytes=run_bytes) == (1001, 3)
  data, _ = check(p, contigs, b''.join(c[0] for c in chunks))
  q = str(tmp_path / 'q.bam')
  assert write(eng, q, contigs, chunks) == (1001, 1)
  assert open(q, 'rb').read() == data and open(q + '.bai', 'rb').read() == open(p + '.bai', 'rb').read()


# ---- 5. record-level edges ------------------------------------------------------------------------------------

LETTERS = b'=ACMGRSVTWYHKDBNacmgrsvtwyhkdbn.*'
QUALS = bytes(range(33, 127))


def test_record_edges_in_one_pair(tmp_path, eng):
  rng = random.Random(1)
  contigs = [('e', 100000)]
  t = [
      ('e', [(0, 100, '4=', b'ACGT', b'IIII'), (1, 200, '4=', b'ACGT', b'IIII')]),                    # padded to 254 bytes below
      ('e', [(1, 300, '1=', b'G', b'#'), (1, 310, '7=', b'ACGTNac', b'!"#$%&\'')]),                     # L = 1 and odd L on strand 1
      ('e', [(1, 400, '%d=' % len(LETTERS), LETTERS, QUALS[:len(LETTERS)]), (0, 450, '%d=' % len(LETTERS), LETTERS, QUALS[-len(LETTERS):])]),
      ('e', [(0, 500, '94=', seq_of(rng, 94), QUALS), (1, 520, '94=', seq_of(rng, 94), QUALS[::-1])]),  # qualities '!' .. '~'
      ('e', [(0, 600, '10=', b'A' * 10, b'I' * 10), (1, 600, '3=2D5=', b'C' * 8, b'I' * 8)]),           # mates at one position
      ('e', [(1, 700, '5=', b'G' * 5, b'I' * 5), (1, 700, '5=', b'T' * 5, b'I' * 5)]),
      ('e', [(0, 800, '2=1X2=', b'ACGTA', b'IIIII'), (1, 803, '>802:6I', b'ACGTAC', b'IIIIII')]),       # a mate inside an insertion
  ]
  fq1, _ = S.fastq(t)
  pad = [255 - len(fq1.split(b'\n')[0])] + [0] * (len(t) - 1)
  fq1, fq2 = S.fastq(t, pad=pad)
  assert len(fq1.split(b'\n')[0]) == 255                            # '@' + a name of exactly 254 bytes
  p = str(tmp_path / 'r.bam')
  assert write(eng, p, contigs, [(fq1, fq2)]) == (14, 1)
  _, recs = check(p, contigs, fq1, fq2)
  by_name = {}
  for r in recs:
    by_name.setdefault(int(r[36:36 + r[12] - 1].split(b'|')[0].rsplit(b':', 1)[1]), []).append(r)
  flag_tlen = lambda r: (struct.unpack_from('<I', r, 16)[0] >> 16, struct.unpack_from('<i', r, 32)[0])
  # mates at one position: file 1 first in the file, TLEN positive on file 1's record, negative on file 2's
  for k in (4, 5):
    (f1, t1), (f2, t2) = map(flag_tlen, by_name[k])
    assert f1 & 0x40 and f2 & 0x80 and t1 > 0 and t2 == -t1
  # a 255-byte name is an error naming the record: the 4th template of the chunk, file 1
  bad = list(t)
  fq1, fq2 = S.fastq(bad, pad=[0, 0, 0, 255 - len(S.fastq(bad)[0].split(b'\n')[12]) + 1, 0, 0, 0])
  assert [len(l) for l in fq1.split(b'\n')[0:-1:4]][3] == 256
  from mitty_b200.engine import BamWriter
  bw = BamWriter(eng, str(tmp_path / 'x.bam'), str(tmp_path / 'x.bam.bai'), contigs, S.header_text(contigs, 'S'), 'S')
  try:
    with pytest.raises(ValueError) as e:
      bw.add(np.frombuffer(fq1, np.uint8), np.frombuffer(fq2, np.uint8))
    assert e.value.args[1:3] == (0, 3) and '254' in e.value.args[3]
  finally:
    bw.abort()
  assert sorted(os.listdir(str(tmp_path))) == ['r.bam', 'r.bam.bai']


# ---- 6. contigs BAM cannot address or BAI cannot index -----------------------------------------------------------

def test_contig_of_2_31_bases_is_rejected_before_any_file(tmp_path, eng):
  from mitty_b200.engine import BamWriter, write_sorted_bam
  for length in (1 << 31, (1 << 32) + 5):
    contigs = [('1', 1000), ('huge', length)]
    with pytest.raises(ValueError, match='huge'):
      BamWriter(eng, str(tmp_path / 'x.bam'), str(tmp_path / 'x.bam.bai'), contigs, S.header_text(contigs, 'S'), 'S')
    with pytest.raises(ValueError, match='huge'):
      write_sorted_bam(str(tmp_path / 'y.bam'), str(tmp_path / 'y.bam.bai'), contigs, S.header_text(contigs, 'S'), b'')
    assert os.listdir(str(tmp_path)) == []


def test_records_past_2_29_without_an_index(tmp_path, eng):
  """A contig of 2^31 - 1 bases: POS, PNEXT and TLEN near their int32 limits, bins past 2^29 whose SAM spec value
  exceeds 16 bits (from 997 048 320 on) keep their low 16 bits; no index is written."""
  rng = random.Random(31)
  top = (1 << 31) - 1
  contigs = [('1', 1000), ('huge', top)]
  edges = S.bin_edge_spans(top, shifts=(14, 26)) + [(997048320 - 1, 1), (997048320, 1), (1 << 29, 1), ((1 << 29) - 1, 2)]
  rng.shuffle(edges)
  templates = [('huge', [read(rng, *edges[i]), read(rng, *edges[i - 1])]) for i in range(len(edges))]
  templates.append(('huge', [read(rng, 0, 5, 0), read(rng, top - 5, 5, 1)]))        # TLEN 2^31 - 1
  fq1, fq2 = S.fastq(templates)
  p = str(tmp_path / 'h.bam')
  assert write(eng, p, contigs, [(fq1, fq2)], bai=False)[0] == 2 * len(templates)
  _, recs = check(p, contigs, fq1, fq2, bai=False)
  # guard: records past 2^29 and past the 16-bit bin, one ending on the last base, the largest TLEN
  full = [S.reg2bin(p0, p0 + max(sp, 1)) for p0, sp in edges]
  assert max(full) > 0xFFFF and max(p0 for p0, _ in edges) >= 1 << 30
  assert max(struct.unpack_from('<i', r, 32)[0] for r in recs) == top
  assert passes(contigs) == 5


def test_no_index_for_a_contig_past_the_bai_limit(tmp_path, monkeypatch, caplog):
  """process_multi_threaded writes no .bai (and removes a stale one) when a contig is longer than
  BAI_MAX_LEN; the limit is lowered here so that a small FASTA takes that branch."""
  import mitty_b200.benchmarking.god_aligner as ga
  from mitty_b200 import synth
  from tests import helpers as H
  wl = synth.edge_workload()
  fa, _, _ = synth.write_workload(wl, str(tmp_path / 'edge'))
  contigs = [(n, int(s.shape[0])) for n, s in wl['contigs']]
  assert max(l for _, l in contigs) > 1000
  monkeypatch.setattr(ga, 'BAI_MAX_LEN', 1000)
  bam = str(tmp_path / 'n.bam')
  open(bam + '.bai', 'wb').write(b'stale')
  f1, f2 = (os.path.join(H.GOLDEN, n) for n in ('edge.r1.fq.gz', 'edge.r2.fq.gz'))
  with caplog.at_level(logging.WARNING, logger=ga.__name__):
    ga.process_multi_threaded(fa, bam, f1, f2, threads=2)
  assert any('2^29' in r.getMessage() for r in caplog.records)
  check(bam, contigs, H.golden_fastq('edge.r1.fq.gz'), H.golden_fastq('edge.r2.fq.gz'), bai=False)
