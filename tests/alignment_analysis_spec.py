"""Independent pure-Python specification of alignment-analysis (struct + re + numpy): an aligner's BAM scored against
the truth in Mitty's qnames.  The BGZF parser, the record walk and the BAM builder are those of
tests/read_model_spec.py; this module adds the header's reference names, the scoring rules and a qname builder.

Every record in file order; the first malformed one (framing, overrun or the rules' errors below) is reported:
  skip      flag & 0x900: counted as skipped, nothing else
  read      index 1 iff (flag & 0xC1) == 0x81, else 0; its qname fields are 3 + 5 * index .. + 4
  errors    17 refID < -1 or >= n_ref; 15 fewer than 8 fields, strand not 0 / 1, pos / v_list entry / '>p:'
            offset not an integer, CIGAR not (digits + one of MIDNSHP=X)+; 16 read 2 with fewer than 13 fields
  column    unmapped (flag & 0x4 or refID -1) = C - 1; wrong chrom = C - 2; else clamp(d, -max_d, max_d) + max_d
  d         (POS - lead(aligned CIGAR)) - (pos - 1 - lead(qname CIGAR)), lead = leading S / H / I (P skipped)
"""
import re
import struct

import numpy as np

from tests.read_model_spec import SpecError, bgzf, header, members, record, records  # noqa: F401 (re-exported for the tests)

COUNTERS = ('records', 'analysed', 'skipped', 'unmapped', 'wrong_chrom', 'exact', 'clamped', 'strand_mismatch', 'no_variant_reads',
            'variant_entries')
CIGAR_OPS = 'MIDNSHP=X'
_INT = re.compile(rb'-?[0-9]+')
_CIGAR = re.compile(rb'(?:[0-9]+[MIDNSHP=X])+')
_OP = re.compile(rb'([0-9]+)([MIDNSHP=X])')


class _NotMitty(Exception):
  pass


def _int(b):
  """A decimal integer with an optional '-', at most 2^40 in magnitude (the device parser's bound)."""
  if not _INT.fullmatch(b) or abs(int(b)) > 1 << 40:
    raise _NotMitty(b)
  return int(b)


def header_info(raw):
  """-> (offset of the first record, [reference name up to its NUL]) of an inflated BAM stream."""
  if raw[:4] != b'BAM\x01':
    raise SpecError('offset', 0, 'not a BAM file')
  u = 8 + struct.unpack_from('<i', raw, 4)[0]
  n_ref = struct.unpack_from('<i', raw, u)[0]
  u += 4
  names = []
  for _ in range(n_ref):                            # l_name, name (NUL-terminated), l_ref
    l_name = struct.unpack_from('<i', raw, u)[0]
    names.append(raw[u + 4:u + 4 + l_name].split(b'\0', 1)[0])
    u += 8 + l_name
  return u, names


def lead(ops):
  """Bases before the alignment start: the leading run of S (4), H (5) and I (1) ops, P (6) skipped."""
  n = 0
  for length, op in ops:
    if op in (1, 4, 5):
      n += length
    elif op != 6:
      break
  return n


def qname_ops(cigar):
  """The (length, op code) list of a qname CIGAR; '>p:nI' is its plain form nI."""
  if cigar[:1] == b'>':
    i = cigar.rfind(b':')
    if i < 1:
      raise _NotMitty(cigar)
    _int(cigar[1:i])
    cigar = cigar[i + 1:]
  if not _CIGAR.fullmatch(cigar):
    raise _NotMitty(cigar)
  return [(_int(n), CIGAR_OPS.index(op.decode())) for n, op in _OP.findall(cigar)]


def score(rec, names, max_d):
  """-> None (skipped) or (column, mapq, v_list, d or None, strand mismatch); raises SpecError for 15-17."""
  ref, pos, l_name, mapq = struct.unpack_from('<iiBB', rec, 4)
  n_cig, flag = struct.unpack_from('<HH', rec, 16)
  if flag & 0x900:
    return None
  if ref < -1 or ref >= len(names):
    raise SpecError('record', None, 'refID out of range')
  f = rec[36:36 + l_name].split(b'\0', 1)[0].split(b'|')
  i = 1 if flag & 0xC1 == 0x81 else 0
  if len(f) < 3 + 5 * i + 5:
    raise SpecError('record', None, 'not a Mitty qname' if len(f) < 8 else 'no read for this mate')
  strand, qpos, _, cigar, vl = f[3 + 5 * i:8 + 5 * i]
  try:
    strand, qpos = _int(strand), _int(qpos)
    if strand not in (0, 1):
      raise _NotMitty(strand)
    truth = qpos - 1 - lead(qname_ops(cigar))
    v_list = [_int(v) for v in vl.split(b',') if v]
  except _NotMitty:
    raise SpecError('record', None, 'not a Mitty qname')
  C = 2 * max_d + 3
  if flag & 0x4 or ref == -1:
    return C - 1, mapq, v_list, None, False
  if names[ref] != f[1]:
    return C - 2, mapq, v_list, None, False
  ops = [(x >> 4, x & 15) for x in struct.unpack_from('<%dI' % n_cig, rec, 36 + l_name)]
  d = pos - lead(ops) - truth
  return min(max(d, -max_d), max_d) + max_d, mapq, v_list, d, (flag >> 4 & 1) != strand


def analyse(recs, names, max_d=200, max_size=50):
  """The rules over a list of record byte strings -> dict of mq, vsize and the counters."""
  C = 2 * max_d + 3
  mq = np.zeros((256, C), dtype=np.uint64)
  vs = np.zeros((2 * max_size + 4, C), dtype=np.uint64)
  c = dict.fromkeys(COUNTERS, 0)
  c['records'] = len(recs)
  for k, rec in enumerate(recs):
    try:
      s = score(rec, names, max_d)
    except SpecError as e:
      raise SpecError('record', k, str(e).split(': ', 1)[1])
    if s is None:
      c['skipped'] += 1
      continue
    col, q, v_list, d, strand_bad = s
    c['analysed'] += 1
    c['unmapped'] += col == C - 1
    c['wrong_chrom'] += col == C - 2
    c['exact'] += d == 0
    c['clamped'] += d is not None and abs(d) > max_d
    c['strand_mismatch'] += strand_bad
    c['no_variant_reads'] += not v_list
    c['variant_entries'] += len(v_list)
    mq[q, col] += 1
    for v in v_list:
      vs[min(max(v, -max_size - 1), max_size + 1) + max_size + 1, col] += 1
    if not v_list:
      vs[-1, col] += 1
  out = {'mq': mq, 'vsize': vs}
  out.update(c)
  return out


def analysis(data, max_d=200, max_size=50):
  """The scores of a BGZF BAM file's bytes.  As on the device, the first malformed thing in stream order is
  reported: a bad member ends the stream before it, a bad record ends the records before it."""
  try:
    raw, member_err = b''.join(r for _, r in members(data)), None
  except SpecError as e:
    raw, member_err = b''.join(r for _, r in members(data[:e.where])), e
  try:
    u, names = header_info(raw)
  except (SpecError, struct.error):
    u, names = len(raw) + 1, None
    if not member_err:
      raise
  if u > len(raw) and member_err:                   # the stream ends inside the header
    raise member_err
  try:
    recs, rec_err = records(raw), None
  except SpecError as e:
    if e.kind != 'record':
      raise
    for _ in range(e.where):                        # the records before the bad one
      u += 4 + struct.unpack_from('<i', raw, u)[0]
    recs, rec_err = records(raw[:u]), e
  res = analyse(recs, names, max_d, max_size)
  if member_err:
    raise member_err
  if rec_err:
    raise rec_err
  return res


def qname(chrom=b'c', reads=((0, 1, 4, b'4=', b''),), serial=b'S:0:0:1', cpy=b'0'):
  """A Mitty qname: reads = [(strand, pos, rlen, cigar, v_list)] in file order; fields are bytes or ints."""
  b = lambda x: x if isinstance(x, bytes) else str(x).encode()  # noqa: E731
  return b'|'.join([serial, chrom, cpy] + [b(x) for r in reads for x in r])
