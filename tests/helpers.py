"""Shared test fixtures: the reference's tiny example, golden-vector access, workload plumbing."""
import gzip
import hashlib
import json
import os

import numpy as np

import oracle
from mitty_b200 import synth
from mitty_b200.lib import vcfio
from mitty_b200.readmodels import load_model

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, 'golden')

# The reference's tiny fixture (mitty/test/data/tiny.fasta, tiny.vcf, tiny.whole.bed, tiny.8-14.bed),
# restated inline: 25 bp of sequence and five variants of sample g0_s0.
TINY_SEQ = 'ATGACGTATCCAAGGAGGCGTTACC'
TINY_VCF = (
  '##fileformat=VCFv4.1\n'
  '##contig=<ID=1,length=23>\n'
  '##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype">\n'
  '#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tg0_s0\n'
  '1\t5\t.\tC\tT\t100\tPASS\t.\tGT\t0|1\n'
  '1\t8\t.\tA\tATTT\t100\tPASS\t.\tGT\t0|1\n'
  '1\t11\t.\tCAA\tC\t100\tPASS\t.\tGT\t0|1\n'
  '1\t14\t.\tG\tT\t100\tPASS\t.\tGT\t1|0\n'
  '1\t20\t.\tGTTAC\tG\t100\tPASS\t.\tGT\t1|1\n')
FLAWED_TINY_VCF = (
  '##fileformat=VCFv4.1\n'
  '##contig=<ID=tiny,length=51>\n'
  '##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype">\n'
  '#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tg0_s0\n'
  '1\t5\t.\tCGT\tCTT\t100\tPASS\t.\tGT\t0|1\n'
  '1\t10\t.\tCCA\tCC\t100\tPASS\t.\tGT\t0|1\n'
  '1\t15\t.\tGA\tGAT\t100\tPASS\t.\tGT\t0|1\n')


def write_tiny(tmp_path, gz=False):
  """-> dict of paths for the tiny fixture files."""
  p = {}
  p['fasta'] = str(tmp_path / 'tiny.fasta')
  with open(p['fasta'], 'w') as fp:
    fp.write('>1\n' + TINY_SEQ + '\n')
  for name, text in (('vcf', TINY_VCF), ('flawed', FLAWED_TINY_VCF)):
    p[name] = str(tmp_path / ('{}.vcf{}'.format(name, '.gz' if gz else '')))
    if gz:
      with gzip.open(p[name], 'wt') as fp:
        fp.write(text)
    else:
      with open(p[name], 'w') as fp:
        fp.write(text)
  p['whole_bed'] = str(tmp_path / 'tiny.whole.bed')
  with open(p['whole_bed'], 'w') as fp:
    fp.write('1\t0\t23')
  p['bed_8_14'] = str(tmp_path / 'tiny.8-14.bed')
  with open(p['bed_8_14'], 'w') as fp:
    fp.write('1\t8\t14')
  return p


_golden = None


def golden():
  global _golden
  if _golden is None:
    with open(os.path.join(GOLDEN, 'golden.json')) as fp:
      _golden = json.load(fp)
  return _golden


def golden_fastq(name):
  with gzip.open(os.path.join(GOLDEN, name), 'rb') as fp:
    return fp.read()


def sha256(b):
  return hashlib.sha256(b).hexdigest()


def oracle_cv(vl):
  """VariantList (product host arrays) -> oracle.CopyVariants (same arrays, no arithmetic)."""
  return oracle.CopyVariants(vl.pos, vl.op, vl.oplen, (vl.alt_pool, vl.alt_off))


def workload_regions(wl):
  """In-memory workload -> region dicts with reference bytes and per-copy variant arrays."""
  contigs = dict(wl['contigs'])
  tables = {t.chrom: t for t in wl['tables']}
  out = []
  for region in wl['regions']:
    chrom, s, e = region
    r = vcfio.from_variant_table(tables[chrom], region)
    r['ref'] = np.ascontiguousarray(contigs[chrom][s:e])
    out.append(r)
  return out


def oracle_regions(regions):
  return [{'region': r['region'], 'ref': r['ref'], 'v': [oracle_cv(v) for v in r['v']]} for r in regions]


def model(name):
  return load_model(name)


def dense_variant_region(seed, alt_n=True):
  """A 6 kb contig with N / IUPAC / soft-masked bytes and a variant set built to stress the greedy skip
  rule (rpc.py:55): long deletions that swallow runs of later variants, chains of overlapping deletions,
  several records at one POS, non-ACGT bytes in ALT alleles.  seed 1..4 sets the density and the longest
  deletion.  alt_n=False puts Y where the ALT alleles would have N (same positions and lengths), so that
  reads are not dropped by the N filter.  -> (region bytes, BED start, VariantList, number of records)."""
  rs = np.random.RandomState(seed)
  n = 6000
  ref = synth.synth_contig(n, seed=100 + seed)
  ref[1000:1100] = ord('N'); ref[3000] = ord('R'); ref[3500:3503] = ord('n')
  bed_start = 40
  recs = []
  for _ in range([400, 1500, 3000, 800][seed - 1]):
    pos = int(rs.randint(1, n - 560))                 # no deletion reaches the region end
    kind = rs.randint(0, 3)
    r0 = chr(ref[pos - 1]).upper()
    r0 = r0 if r0 in 'ACGT' else 'A'
    if kind == 0:
      recs.append((pos, r0, ('ACGTN' if alt_n else 'ACGTY')[rs.randint(0, 5)], 'X', 0))
    elif kind == 1:
      ol = int(rs.randint(1, 40))
      recs.append((pos, r0, r0 + ''.join(('ACGTRN' if alt_n else 'ACGTRY')[i] for i in rs.randint(0, 6, size=ol)), 'I', ol))
    else:
      ol = int(rs.randint(1, [8, 30, 50, 200][seed - 1]))
      recs.append((pos, 'A' * (ol + 1), 'A', 'D', ol))
  recs.sort(key=lambda t: t[0])                       # stable: records at one POS keep their order
  vl = vcfio.VariantList.from_variants([vcfio.Variant(*t) for t in recs])
  return np.ascontiguousarray(ref[bed_start:n - 300]), bed_start, vl, len(recs)


# ---- god-aligner style round trip -------------------------------------------------------------------

class HaplotypeIndex(object):
  """Independent re-derivation of reads from their qname, the way Mitty's god-aligner trusts it
  (mitty/benchmarking/god_aligner.py:141-183 over readgenerate.parse_qname): POS is a REFERENCE
  coordinate, so the read is located through a reference->haplotype map built from the oracle's
  node list, then the CIGAR is walked over reference and haplotype together."""

  def __init__(self, ref, ref_start_pos, cv):
    self.nodes = oracle.create_node_list(ref, ref_start_pos, cv)
    self.p_min = self.nodes[0][0]
    self.hap = ''.join(n[4] for n in self.nodes)
    self.ref = ref.tobytes().decode() if isinstance(ref, np.ndarray) else ref
    self.ref_start = ref_start_pos
    # reference position -> sample position for '=' and 'X' nodes
    self.eq_pr = np.array([n[1] for n in self.nodes if n[2] in '=X'], dtype=np.int64)
    self.eq_ps = np.array([n[0] for n in self.nodes if n[2] in '=X'], dtype=np.int64)
    self.ins = {n[1]: n for n in self.nodes if n[2] == 'I'}   # keyed by pr

  def ref_to_samp(self, pos):
    k = np.searchsorted(self.eq_pr, pos, side='right') - 1
    return int(self.eq_ps[k] + (pos - self.eq_pr[k]))

  def check(self, info, seq):
    """info: ReadInfo from parse_qname; seq: the FASTQ sequence as written. Returns None or an error string."""
    import re
    comp = str.maketrans('ATCGN', 'TAGCN')
    fwd = seq.translate(comp)[::-1] if info.strand else seq    # god_aligner.py:163-166
    if info.special_cigar is not None:
      m = re.match(r'>(\d+):(\d+)I', info.special_cigar)
      node = self.ins.get(info.pos + 1)
      if node is None:
        return 'no insertion after pos {}'.format(info.pos)
      off, n = int(m.group(1)), int(m.group(2))
      return None if node[4][off:off + n] == fwd else 'inside-insertion read mismatch'
    ops = re.findall(r'(\d+)(\D)', info.cigar)
    if sum(int(c) for c, o in ops if o != 'D') != info.rlen or len(fwd) != info.rlen:
      return 'cigar length != rlen'
    rp, i = info.pos, 0
    first = True
    for c, o in ops:
      c = int(c)
      if o == '=':
        if self.ref[rp - self.ref_start:rp - self.ref_start + c] != fwd[i:i + c]:
          return '= segment differs from the reference at {}'.format(rp)
        rp += c; i += c
      elif o == 'X':
        s = self.ref_to_samp(rp) - self.p_min
        if self.hap[s:s + c] != fwd[i:i + c]:
          return 'X base differs from the haplotype at {}'.format(rp)
        rp += c; i += c
      elif o == 'I':
        node = self.ins.get(rp)
        if node is None:
          return 'no insertion at {}'.format(rp)
        ins = node[4]
        if (ins[len(ins) - c:] if first else ins[:c]) != fwd[i:i + c]:
          return 'inserted bases differ at {}'.format(rp)
        i += c
      elif o == 'D':
        rp += c
      else:
        return 'unexpected op ' + o
      first = False
    return None


def roundtrip_fastq(f1, f2, index_for):
  """Every read of a FASTQ pair re-derived from its qname. index_for(chrom, cpy) -> HaplotypeIndex.
  Returns (reads checked, list of errors)."""
  from mitty_b200.simulation.readgenerate import parse_qname
  errs, n = [], 0
  for buf in (f1, f2):
    lines = buf.decode().split('\n')
    which = 0 if buf is f1 else 1
    for k in range(0, len(lines) - 1, 4):
      infos = parse_qname(lines[k][1:])
      info = infos[which]
      e = index_for(info.chrom, info.cpy).check(info, lines[k + 1])
      n += 1
      if e:
        errs.append((lines[k], e))
  return n, errs


def feed_interleaved(paths, datas, piece=256 << 10):
  """One writer for a FIFO pair, as a tool that writes mate 1 and then mate 2 of each template in one loop:
  ``piece`` bytes of file 1, then of file 2, and so on.  A reader that waits for one file to fill its buffer
  before it reads the other blocks this writer on the other pipe."""
  fps = [open(p, 'wb') for p in paths]          # each open blocks until the reader has opened that FIFO
  for off in range(0, max(len(d) for d in datas), piece):
    for fp, d in zip(fps, datas):
      if off < len(d):
        fp.write(d[off:off + piece])
        fp.flush()
  for fp in fps:
    fp.close()
