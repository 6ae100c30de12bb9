"""Host-side front half of the haplotype builder: BED / VCF / FASTA -> per-region, per-copy
variant arrays.  Mirrors ``mitty/lib/vcfio.py`` (reference) function for function:

* ``read_bed``            <- vcfio.py:45-46   (0-based half-open, file order preserved)
* ``load_variant_file``   <- vcfio.py:51-64   (records overlapping each BED region, htslib rule)
* ``split_copies``        <- vcfio.py:67-102  (ploidy = len(GT) of the FIRST record; empty -> 2)
* ``parse`` / ``Variant`` <- vcfio.py:19-33,105-126  (X / I / D classification, ValueError on
                                                      complex variants)

pysam/htslib is not a dependency: VCF text (plain or gzip/bgzip) is parsed here, and the htslib
region-overlap rule (a record at 1-based POS occupies 0-based [POS-1, POS-1+len(REF)) and is
returned iff that overlaps [start, stop)) is applied with numpy (the reference's own
test_vcfio.py:9-18 pins it: deletion at 11 is returned for [8,14), insertion at 8 is not).

The per-copy result is a ``VariantList``: flat numpy arrays ready for the C-ABI
(``mg_copy_build``), which also behaves like the reference's ``list`` of ``Variant`` objects.
"""
import ctypes as C
import os
import gzip
import re
import time
import logging
import threading

import numpy as np

logger = logging.getLogger(__name__)


class Variant(object):
  """Same fields and tuple() as the reference's Variant (vcfio.py:19-33)."""
  __slots__ = ('pos', 'ref', 'alt', 'cigarop', 'oplen')

  def __init__(self, pos, ref, alt, cigarop, oplen):
    self.pos, self.ref, self.alt, self.cigarop, self.oplen = pos, ref, alt, cigarop, oplen

  def tuple(self):
    return self.pos, self.ref, self.alt, self.cigarop, self.oplen

  def __repr__(self):
    return self.tuple().__repr__()


class VariantList(object):
  """Variants on one chromosome copy, as flat arrays (pos, op, oplen, pooled REF/ALT bytes)."""
  __slots__ = ('pos', 'op', 'oplen', 'alt_pool', 'alt_off', 'ref_pool', 'ref_off')

  def __init__(self, pos, op, oplen, alt_pool, alt_off, ref_pool=None, ref_off=None):
    self.pos = np.ascontiguousarray(pos, dtype=np.int64)
    self.op = np.ascontiguousarray(op, dtype=np.uint8)
    self.oplen = np.ascontiguousarray(oplen, dtype=np.int64)
    self.alt_pool = np.ascontiguousarray(alt_pool, dtype=np.uint8)
    self.alt_off = np.ascontiguousarray(alt_off, dtype=np.int64)
    self.ref_pool, self.ref_off = ref_pool, ref_off

  @classmethod
  def from_variants(cls, vl):
    """From a list of Variant-like objects (pos, ref, alt, cigarop, oplen)."""
    alts = [v.alt.encode() for v in vl]
    refs = [v.ref.encode() for v in vl]
    alt_off = np.zeros(len(vl) + 1, dtype=np.int64); np.cumsum([len(a) for a in alts], out=alt_off[1:])
    ref_off = np.zeros(len(vl) + 1, dtype=np.int64); np.cumsum([len(a) for a in refs], out=ref_off[1:])
    return cls([v.pos for v in vl], np.frombuffer(''.join(v.cigarop for v in vl).encode(), dtype=np.uint8),
               [v.oplen for v in vl], np.frombuffer(b''.join(alts), dtype=np.uint8), alt_off,
               np.frombuffer(b''.join(refs), dtype=np.uint8), ref_off)

  def __len__(self):
    return int(self.pos.shape[0])

  def __getitem__(self, i):
    if isinstance(i, slice):
      return [self[j] for j in range(*i.indices(len(self)))]
    if i < 0:
      i += len(self)
    if not 0 <= i < len(self):
      raise IndexError(i)
    ref = '' if self.ref_pool is None else self.ref_pool[self.ref_off[i]:self.ref_off[i + 1]].tobytes().decode()
    alt = self.alt_pool[self.alt_off[i]:self.alt_off[i + 1]].tobytes().decode()
    return Variant(int(self.pos[i]), ref, alt, chr(self.op[i]), int(self.oplen[i]))

  def __iter__(self):
    return (self[i] for i in range(len(self)))


def read_bed(bed_fname):
  """BED -> [(chrom, start, end)], whitespace split, file order preserved (vcfio.py:45-46)."""
  out = []
  with open(bed_fname, 'r') as fp:
    for line in fp.readlines():
      x = line.split()
      out.append((x[0], int(x[1]), int(x[2])))
  return out


def _open_bytes(fname):
  with open(fname, 'rb') as fp:
    magic = fp.read(2)
  if magic == b'\x1f\x8b':
    with gzip.open(fname, 'rb') as fp:  # also reads bgzip (concatenated gzip members)
      return fp.read()
  with open(fname, 'rb') as fp:
    return fp.read()


class _Contig(object):
  """Records of one contig as arrays over the file's bytes (no per-record Python objects)."""
  __slots__ = ('pos', 'reflen', 'rs', 're', 'as_', 'ae', 'gt', 'ploidy', 'exotic', 'slow', 'ls', 'le', 'f9e', 'ss', 'se', 'p0', 'is_sorted', 'max_reflen')

  def __init__(self, pos, rs, re_, as_, ae, gt, ploidy, exotic, slow, lines=None):
    self.pos, self.rs, self.re, self.as_, self.ae = pos, rs, re_, as_, ae
    # byte ranges of the whole line, of its first nine columns and of the sample column (filter-variants)
    self.ls, self.le, self.f9e, self.ss, self.se = lines if lines is not None else (None,) * 5
    self.reflen = re_ - rs
    self.gt, self.ploidy, self.exotic, self.slow = gt, ploidy, exotic, slow
    self.p0 = None                                    # the fetch index (0-based starts, sortedness, longest REF), made on first use

  def fetch_index(self):
    if self.p0 is None:
      self.p0 = self.pos - 1
      self.is_sorted = bool(self.p0.size < 2 or (self.p0[1:] >= self.p0[:-1]).all())
      self.max_reflen = int(self.reflen.max()) if self.reflen.size else 1
    return self.p0

  def merged(self, o):
    n = self.pos.size
    slow = dict(self.slow); slow.update({k + n: v for k, v in o.slow.items()})
    w = max(self.gt.shape[1], o.gt.shape[1])
    def widen(g):
      out = np.full((g.shape[0], w), -2, dtype=np.int8); out[:, :g.shape[1]] = g
      return out
    cat = np.concatenate
    return _Contig(cat([self.pos, o.pos]), cat([self.rs, o.rs]), cat([self.re, o.re]), cat([self.as_, o.as_]), cat([self.ae, o.ae]),
                   cat([widen(self.gt), widen(o.gt)]), cat([self.ploidy, o.ploidy]), cat([self.exotic, o.exotic]), slow,
                   tuple(cat([a, b]) for a, b in zip((self.ls, self.le, self.f9e, self.ss, self.se), (o.ls, o.le, o.f9e, o.ss, o.se))))


def _gt_tuple(fmt, s):
  if fmt != 'GT':
    s = s.split(':')[fmt.split(':').index('GT')]
  return tuple(None if g == '.' else int(g) for g in s.replace('/', '|').split('|'))


VCF_PIECE_BYTES = 4 << 20      # a VCF body larger than two of these is parsed in pieces by threads (1.19 -> 0.23 s for 1.2 M records on 8 cores)


class VcfTable(object):
  """All records of one sample, grouped by contig, parsed with numpy over the raw bytes (a 4 M-record
  WGS call set in seconds; the reference walks pysam records one by one, vcfio.py:59-62).

  Per contig (``_Contig``): pos int64[n]; byte ranges of REF and ALT in ``self.buf``; gt int8[n, P]
  (allele index per GT column, -1 for '.', -2 beyond the record's ploidy); ploidy int8[n].  Records
  the array path does not cover -- multi-allelic ALT, FORMAT not starting with GT, allele indices
  of more than one digit -- are parsed individually into ``slow`` {record: (ref, alleles, gt)}.
  """

  def __init__(self, fname, sample):
    if str(fname).endswith('bcf'):
      raise NotImplementedError('BCF input needs htslib; convert to VCF text (plain or gzip)')
    data = _open_bytes(fname)
    self.buf = buf = np.frombuffer(data, dtype=np.uint8)
    self.data = data
    self.contigs = {}
    self.sample = sample
    h = 0 if data.startswith(b'#CHROM') else data.find(b'\n#CHROM') + 1
    if h == 0 and not data.startswith(b'#CHROM'):
      raise ValueError('No #CHROM header line in {}'.format(fname))
    he = data.find(b'\n', h)
    he = len(data) if he < 0 else he
    hdr = data[h:he].decode().rstrip('\r').split('\t')
    if sample not in hdr[9:]:
      raise ValueError('Sample {} not in VCF (samples: {})'.format(sample, hdr[9:]))
    col = 9 + hdr[9:].index(sample)
    self.header_end = h                                                 # the '##' meta lines are data[:h]
    # contigs the header declares (##contig=<ID=...>): with the contigs seen in the body these are the
    # names an indexed fetch accepts; pysam raises ValueError for any other (vcfio.py:62)
    self.header_contigs = set(m.decode() for m in re.findall(rb'^##contig=<(?:[^>\n]*,)?ID=([^,>\n]+)', data[:h], flags=re.M))
    body = min(he + 1, len(data))
    # large files: the body is cut at line starts into pieces parsed by threads (numpy releases the GIL in the
    # scans, searches and gathers that make up the parser); a contig met again in a later piece is merged
    n_pieces = 1
    if len(data) - body > 2 * VCF_PIECE_BYTES:
      n_pieces = max(1, min(os.cpu_count() or 1, 16, (len(data) - body) // VCF_PIECE_BYTES))
    cuts = [body]
    for k in range(1, n_pieces):
      at = data.find(b'\n', body + (len(data) - body) * k // n_pieces)
      if at < 0:
        break
      if at + 1 > cuts[-1]:
        cuts.append(at + 1)
    cuts.append(len(data))
    ranges = [(lo, hi) for lo, hi in zip(cuts[:-1], cuts[1:]) if hi > lo]
    if len(ranges) > 1:
      from concurrent.futures import ThreadPoolExecutor
      with ThreadPoolExecutor(len(ranges)) as ex:
        parts = list(ex.map(lambda r: self._parse_range(r[0], r[1], col, fname), ranges))
    else:
      parts = [self._parse_range(lo, hi, col, fname) for lo, hi in ranges]
    for part in parts:
      for name, c in part:
        self.contigs[name] = self.contigs[name].merged(c) if name in self.contigs else c

  def _parse_range(self, body, stop, col, fname):
    """The records of data[body:stop] (whole lines) -> [(contig name, _Contig)] in file order.  Byte
    positions in the _Contig arrays are absolute (into self.buf)."""
    data, buf = self.data, self.buf
    out = []
    nl = np.flatnonzero(buf[body:stop] == 10) + body
    starts = np.concatenate([np.array([body], dtype=np.int64), nl + 1])
    ends = np.concatenate([nl, np.array([stop], dtype=np.int64)])
    keep = ends > starts
    starts, ends = starts[keep], ends[keep]
    if starts.size:
      keep = buf[starts] != 35                                           # stray '#' lines
      starts, ends = starts[keep], ends[keep]
      ends = ends - (buf[ends - 1] == 13)                                # CRLF
    tabs = np.flatnonzero(buf[body:stop] == 9) + body
    t0 = np.searchsorted(tabs, starts)
    ntab = np.searchsorted(tabs, ends) - t0
    keep = ntab >= col                                                   # short lines are skipped
    starts, ends, t0, ntab = starts[keep], ends[keep], t0[keep], ntab[keep]
    n = starts.size
    if n == 0:
      return out
    tabs_p = np.concatenate([tabs, np.array([stop], dtype=np.int64)])

    def fs(k):
      return starts if k == 0 else tabs[t0 + k - 1] + 1

    def fe(k):
      return np.where(ntab > k, tabs_p[np.minimum(t0 + k, tabs.size)], ends)

    def gather(s0, ln):
      w = int(ln.max()) if ln.size else 0
      mat = np.zeros((ln.size, w), dtype=np.uint8)
      for k in range(w):
        m = ln > k
        mat[m, k] = buf[s0[m] + k]
      return mat

    # POS
    ps, pe = fs(1), fe(1)
    dig = gather(ps, pe - ps)
    plen = pe - ps
    pos = np.zeros(n, dtype=np.int64)
    for k in range(dig.shape[1]):
      m = plen > k
      d = dig[m, k].astype(np.int64) - 48
      if ((d < 0) | (d > 9)).any():
        raise ValueError('Malformed POS field in {}'.format(fname))
      pos[m] = pos[m] * 10 + d
    rs, re_, as_, ae = fs(3), fe(3), fs(4), fe(4)
    # which records need the per-line path
    commas = np.flatnonzero(buf[body:stop] == 44) + body
    exotic = (np.searchsorted(commas, ae) - np.searchsorted(commas, as_)) > 0
    f8s, f8e = fs(8), fe(8)
    flen = f8e - f8s
    ok_fmt = (flen >= 2) & (buf[f8s] == 71) & (buf[np.minimum(f8s + 1, len(data) - 1)] == 84)
    ok_fmt &= (flen == 2) | (buf[np.minimum(f8s + 2, len(data) - 1)] == 58)
    ss, se = fs(col), fe(col)
    colons = np.flatnonzero(buf[body:stop] == 58) + body
    ci = np.searchsorted(colons, ss)
    cpos = np.concatenate([colons, np.array([stop], dtype=np.int64)])[np.minimum(ci, colons.size)]
    ge = np.minimum(cpos, se)
    glen = ge - ss
    gmat = gather(ss, np.minimum(glen, 15))
    maxp = (gmat.shape[1] + 1) // 2
    gt = np.full((n, max(maxp, 1)), -2, dtype=np.int8)
    simple = (glen % 2 == 1) & (glen <= 15)
    for j in range(maxp):
      m = glen > 2 * j
      c = gmat[m, 2 * j]
      simple[m] &= ((c >= 48) & (c <= 57)) | (c == 46)
      gt[m, j] = np.where(c == 46, -1, c.astype(np.int16) - 48).astype(np.int8)
      if 2 * j + 1 < gmat.shape[1]:
        m2 = glen > 2 * j + 1
        sep = gmat[m2, 2 * j + 1]
        simple[m2] &= (sep == 124) | (sep == 47)
    exotic |= ~ok_fmt | ~simple
    ploidy = ((glen + 1) // 2).astype(np.int16)
    slow_all = {}
    for i in np.flatnonzero(exotic).tolist():
      f = data[starts[i]:ends[i]].decode().split('\t')
      g = _gt_tuple(f[8], f[col])
      slow_all[i] = (f[3], (f[3],) + tuple(f[4].split(',')), g)
      ploidy[i] = len(g)
    # contig runs
    cmat = gather(starts, fe(0) - starts)
    clen = fe(0) - starts
    change = np.ones(n, dtype=bool)
    if n > 1:
      change[1:] = (cmat[1:] != cmat[:-1]).any(axis=1) | (clen[1:] != clen[:-1])
    run0 = np.flatnonzero(change)
    run1 = np.concatenate([run0[1:], np.array([n])])
    for a, b in zip(run0.tolist(), run1.tolist()):
      name = cmat[a, :clen[a]].tobytes().decode()
      slow = {i - a: v for i, v in slow_all.items() if a <= i < b} if slow_all else {}
      c = _Contig(pos[a:b], rs[a:b], re_[a:b], as_[a:b], ae[a:b], gt[a:b], ploidy[a:b], exotic[a:b], slow,
                  (starts[a:b], ends[a:b], f8e[a:b], ss[a:b], se[a:b]))
      out.append((name, c))
    return out

  def fetch(self, contig, start, stop):
    """Indices of records overlapping 0-based [start, stop) -- htslib semantics (vcfio.py:62)."""
    if contig not in self.contigs:
      if contig not in self.header_contigs:
        # pysam: "ValueError: invalid contig `chr1`" -- e.g. a BED that says 'chr1' over a VCF that says '1'.
        # Going on would silently produce variant-free reads with truth qnames.
        raise ValueError('invalid contig `{}`: not in the VCF header (##contig) nor among its records ({})'.format(
          contig, ', '.join(sorted(set(self.contigs) | self.header_contigs)[:8]) or 'no contigs at all'))
      return contig, np.zeros(0, dtype=np.int64)
    c = self.contigs[contig]
    p0 = c.fetch_index()
    if c.is_sorted:
      # records sorted by POS (every indexed VCF): the overlapping ones lie in a window found by two binary searches
      # -- an exome BED of 200 000 targets over a 4 M-record call set would otherwise scan 10^12 elements
      lo = int(np.searchsorted(p0, start - c.max_reflen + 1, side='left'))
      hi = int(np.searchsorted(p0, stop, side='left'))
      if hi <= lo:
        return contig, np.zeros(0, dtype=np.int64)
      return contig, lo + np.flatnonzero(p0[lo:hi] + c.reflen[lo:hi] > start)
    return contig, np.flatnonzero((p0 < stop) & (p0 + c.reflen > start))

  def gt_of(self, contig, i):
    """GT of record i as the tuple pysam would give (None for '.')."""
    c = self.contigs[contig]
    if i in c.slow:
      return c.slow[i][2]
    return tuple(None if g == -1 else int(g) for g in c.gt[i, :c.ploidy[i]])


def _pool(buf, s0, ln):
  off = np.zeros(ln.size + 1, dtype=np.int64)
  np.cumsum(ln, out=off[1:])
  src = np.repeat(s0 - off[:-1], ln) + np.arange(off[-1])
  return (buf[src] if src.size else np.zeros(0, dtype=np.uint8)), off


def _parse_copy_records(table, contig, idx, cpy):
  """Per-record path (vcfio.parse, vcfio.py:105-126) for selections that hold multi-allelic or
  otherwise unusual records."""
  c = table.contigs[contig]
  buf = table.buf
  pos, op, oplen, alts, refs = [], [], [], [], []
  for i in idx.tolist():
    if i in c.slow:
      ref, alleles, gt = c.slow[i]
    else:
      ref = buf[c.rs[i]:c.re[i]].tobytes().decode()
      alleles = (ref, buf[c.as_[i]:c.ae[i]].tobytes().decode())
      gt = table.gt_of(contig, i)
    g = gt[cpy]                            # IndexError on ragged ploidy, like the reference
    if g == 0:                             # not present on this copy (vcfio.py:112)
      continue
    if g is None:
      raise ValueError('Missing GT allele at {}:{}'.format(contig, int(c.pos[i])))
    alt = alleles[g]
    l_r, l_a = len(ref), len(alt)
    if l_r == 1:
      if l_a == 1:
        o, ol = 88, 0                      # 'X'
      else:
        o, ol = 73, l_a - l_r              # 'I'
    elif l_a == 1:
      o, ol = 68, l_r - l_a                # 'D'
    else:
      raise ValueError("Complex variants present in VCF. Please filter or refactor these.")
    pos.append(int(c.pos[i])); op.append(o); oplen.append(ol); alts.append(alt.encode()); refs.append(ref.encode())
  alt_off = np.zeros(len(pos) + 1, dtype=np.int64); np.cumsum([len(a) for a in alts], out=alt_off[1:])
  ref_off = np.zeros(len(pos) + 1, dtype=np.int64); np.cumsum([len(a) for a in refs], out=ref_off[1:])
  return VariantList(pos, np.array(op, dtype=np.uint8), oplen, np.frombuffer(b''.join(alts), dtype=np.uint8), alt_off,
                     np.frombuffer(b''.join(refs), dtype=np.uint8), ref_off)


_EMPTY_VL = VariantList([], np.zeros(0, np.uint8), [], np.zeros(0, np.uint8), np.zeros(1, np.int64), np.zeros(0, np.uint8), np.zeros(1, np.int64))
for _a in (_EMPTY_VL.pos, _EMPTY_VL.op, _EMPTY_VL.oplen, _EMPTY_VL.alt_pool, _EMPTY_VL.alt_off, _EMPTY_VL.ref_pool, _EMPTY_VL.ref_off):
  _a.setflags(write=False)


def parse_copy(table, contig, idx, cpy):
  """vcfio.parse over the records ``idx`` for copy ``cpy`` -> VariantList (vcfio.py:105-126)."""
  if idx.size == 0:
    return _EMPTY_VL                                       # shared: VariantLists are read-only everywhere
  c = table.contigs[contig]
  if c.exotic[idx].any():
    return _parse_copy_records(table, contig, idx, cpy)
  if (c.ploidy[idx] <= cpy).any():
    raise IndexError('tuple index out of range')           # ragged ploidy, like the reference
  g = c.gt[idx, cpy]
  if (g == -1).any():
    raise ValueError('Missing GT allele at {}:{}'.format(contig, int(c.pos[idx[np.flatnonzero(g == -1)[0]]])))
  if (g > 1).any():
    raise IndexError('tuple index out of range')           # allele index beyond the single ALT
  sel = idx[g != 0]                                        # GT 0: not on this copy (vcfio.py:112)
  l_r, l_a = c.reflen[sel], (c.ae - c.as_)[sel]
  if ((l_r > 1) & (l_a > 1)).any():
    raise ValueError("Complex variants present in VCF. Please filter or refactor these.")
  op = np.where(l_r == 1, np.where(l_a == 1, 88, 73), 68).astype(np.uint8)
  oplen = np.where(l_r == 1, l_a - 1, l_r - 1)
  ap, ao = _pool(table.buf, c.as_[sel], l_a)
  rp, ro = _pool(table.buf, c.rs[sel], l_r)
  return VariantList(c.pos[sel], op, oplen, ap, ao, rp, ro)


def split_copies(region, table, contig, idx):
  """One VariantList per chromosome copy; ploidy sniffed from the first record (vcfio.py:67-102)."""
  if idx.size == 0:
    logger.warning('Empty region ({}), assuming diploid'.format(region))
    ploidy = 2
  else:
    ploidy = len(table.gt_of(contig, int(idx[0])))
    logger.debug('Region: {}, ploidy: {}'.format(region, ploidy))
  return {'region': region, 'v': [parse_copy(table, contig, idx, cpy) for cpy in range(ploidy)]}


def load_variant_file(fname, sample, bed_fname):
  """VCF + BED -> [{'region': (chrom, start, end), 'v': [VariantList per copy]}] (vcfio.py:51-64)."""
  table = VcfTable(fname, sample)
  return [split_copies(region, table, *table.fetch(region[0], region[1], region[2]))
          for region in read_bed(bed_fname)]


def prepare_variant_file(fname_in, sample, bed_fname, fname_out, write_mode='w'):
  """filter-variants (vcfio.prepare_variant_file, vcfio.py:128-169): the VCF restricted to one sample
  and to the BED regions, with complex calls removed -- a record is dropped when an allele the sample
  carries has len(REF) > 1 and len(allele) > 1 and differs from REF.  As in the reference, a record
  overlapping two regions is written once per region.  Output is VCF text (gzip if the name ends in
  '.gz'); the meta lines are kept and the column header names only ``sample``."""
  t0 = time.time()
  table = VcfTable(fname_in, sample)
  data = table.data
  out = [data[:table.header_end], ('#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t' + sample + '\n').encode()]
  v_cnt = fltr_cnt = 0
  for region in read_bed(bed_fname):
    contig, idx = table.fetch(region[0], region[1], region[2])
    if idx.size == 0:
      continue
    c = table.contigs[contig]
    cx = (c.reflen[idx] > 1) & ((c.ae - c.as_)[idx] > 1) & (c.gt[idx] == 1).any(axis=1)
    for k in np.flatnonzero(cx & (c.reflen[idx] == (c.ae - c.as_)[idx])).tolist():   # `_v.ref != alt` (vcfio.py:143)
      i = int(idx[k])
      cx[k] = data[c.rs[i]:c.re[i]] != data[c.as_[i]:c.ae[i]]
    for k, i in enumerate(idx.tolist()):
      if i in c.slow:
        ref, alleles, gt = c.slow[i]
        cx[k] = any(len(ref) > 1 and len(alleles[g]) > 1 and alleles[g] != ref for g in gt if g is not None and g < len(alleles))
      elif c.exotic[i]:
        cx[k] = False
    v_cnt += int(idx.size)
    fltr_cnt += int(cx.sum())
    for i in idx[~cx].tolist():
      out.append(data[c.ls[i]:c.f9e[i]] + b'\t' + data[c.ss[i]:c.se[i]] + b'\n')
  blob = b''.join(out)
  if str(fname_out) == '-':                 # `filter-variants ... - | bgzip -c > x.vcf.gz` (examples/reads/run.sh:9)
    import sys
    sys.stdout.buffer.write(blob)
    sys.stdout.buffer.flush()
  elif str(fname_out).endswith('.gz'):
    with gzip.open(fname_out, 'wb') as fp:
      fp.write(blob)
  else:
    with open(fname_out, 'wb') as fp:
      fp.write(blob)
  logger.debug('Processed {} variants'.format(v_cnt))
  logger.debug('Filtered out {} complex variants'.format(fltr_cnt))
  logger.debug('Took {} s'.format(time.time() - t0))
  return v_cnt, fltr_cnt


def from_variant_table(vt, region):
  """Same structure from an in-memory synthetic ``mitty_b200.synth.VariantTable`` (single ALT)."""
  chrom, start, stop = region
  p0 = vt.pos - 1
  reflen = vt.ref_off[1:] - vt.ref_off[:-1]
  altlen = vt.alt_off[1:] - vt.alt_off[:-1]
  sel = (p0 < stop) & (p0 + reflen > start)
  if ((reflen > 1) & (altlen > 1))[sel].any():
    raise ValueError("Complex variants present in VCF. Please filter or refactor these.")
  ploidy = vt.gt.shape[1] if sel.any() else 2
  op = np.where(reflen == 1, np.where(altlen == 1, 88, 73), 68).astype(np.uint8)
  oplen = np.where(reflen == 1, altlen - 1, reflen - 1)
  out = []
  for cpy in range(ploidy):
    idx = np.flatnonzero(sel & (vt.gt[:, cpy] != 0)) if sel.any() else np.zeros(0, dtype=np.int64)
    def pool(p, off):
      ln = (off[1:] - off[:-1])[idx]
      noff = np.zeros(idx.size + 1, dtype=np.int64); np.cumsum(ln, out=noff[1:])
      src = np.repeat(off[:-1][idx] - noff[:-1], ln) + np.arange(noff[-1])
      return p[src] if src.size else np.zeros(0, dtype=np.uint8), noff
    ap, ao = pool(vt.alt_pool, vt.alt_off)
    rp, ro = pool(vt.ref_pool, vt.ref_off)
    out.append(VariantList(vt.pos[idx], op[idx], oplen[idx], ap, ao, rp, ro))
  return {'region': region, 'v': out}


class FastaFile(object):
  """FASTA reader with pysam.FastaFile's fetch(reference=, start=, end=) (readgenerate.py:181,186).
  Sequences come back as uint8 arrays of the file's bytes (case and IUPAC codes preserved).

  Plain files go through the library's native reader (mg_fasta_*: the file is mapped, a fetch is one
  memcpy per line and holds no GIL, so the worker threads of several GPUs fetch at once); gzip'd files
  (and a missing library) through the bytes-level reader below."""

  def __init__(self, fname, native=True):
    self._h = None
    self._lengths = {}
    if native:
      try:
        from mitty_b200 import _lib
        L = _lib.lib()
        h = C.c_void_p()
        if L.mg_fasta_open(str(fname).encode(), C.byref(h)) == 0:
          self._L, self._h = L, h
          name, ln = C.c_char_p(), C.c_int64(0)
          for i in range(L.mg_fasta_n_contigs(h)):
            L.mg_fasta_contig(h, i, C.byref(name), C.byref(ln), None)
            self._lengths.setdefault(name.value.decode(), ln.value)
          return
      except (RuntimeError, OSError, AttributeError):
        self._h = None
    data = _open_bytes(fname)
    self._seqs = {}
    # headers are '>' at a line start; bytes.find runs at memchr speed (a 3 GB genome in a second)
    hdr = []
    h = 0 if data.startswith(b'>') else data.find(b'\n>') + 1
    while h > 0 or (h == 0 and data.startswith(b'>') and not hdr):
      hdr.append(h)
      h = data.find(b'\n>', h) + 1
    bounds = hdr + [len(data)]
    for k, h in enumerate(hdr):
      eol = data.find(b'\n', h)
      if eol < 0:
        eol = len(data)
      name = data[h + 1:eol].split()[0].decode() if eol > h + 1 else ''
      self._seqs.setdefault(name, (min(eol + 1, len(data)), bounds[k + 1]))
    self._data = data
    self._cache = {}
    self._lock = threading.Lock()

  @property
  def references(self):
    return list(self._lengths) if self._h is not None else list(self._seqs)

  def get_reference_length(self, reference):
    """Length of a contig (pysam.FastaFile.get_reference_length)."""
    return self._lengths[reference] if self._h is not None else len(self._contig(reference))

  def close(self):
    if self._h is not None:
      self._L.mg_fasta_close(self._h)
      self._h = None
      self._lengths = {}

  def __del__(self):
    try:
      self.close()
    except Exception:
      pass

  def _contig(self, name):
    with self._lock:   # one worker thread per GPU may fetch concurrently
      if name not in self._cache:
        s, e = self._seqs[name]
        self._cache[name] = np.frombuffer(self._data[s:e].translate(None, b'\r\n'), dtype=np.uint8)
      return self._cache[name]

  def fetch(self, reference=None, start=None, end=None, out=None):
    """out: optional uint8 array (e.g. page-locked) to receive the bases; a view of it is returned."""
    if self._h is None:
      seq = self._contig(reference)[start:end]
      if out is None:
        return seq
      out[:seq.size] = seq
      return out[:seq.size]
    n = self._lengths[reference]                       # KeyError for an unknown contig, as the dict above
    a, b, _ = slice(start, end).indices(n)
    m = max(0, b - a)
    if out is None:
      out = np.empty(m, dtype=np.uint8)
    elif out.size < m or out.dtype != np.uint8 or not out.flags['C_CONTIGUOUS']:
      raise ValueError('FastaFile.fetch: out must be a contiguous uint8 array of at least {} bytes'.format(m))
    if m:
      got = self._L.mg_fasta_fetch(self._h, str(reference).encode(), a, b, C.c_void_p(out.ctypes.data), 4)
      if got != m:
        raise IOError('FASTA fetch of {}:{}-{} returned {} of {} bases'.format(reference, a, b, got, m))
    return out[:m]
