"""Independent pure-Python specification of bam2illumina's counts (struct + zlib + numpy): a general BGZF
parser (any XLEN, the 'BC' subfield located among others, optional FNAME / FCOMMENT / FHCRC), the BAM record
walk, the counting rules, and a builder for arbitrary BAM records and BGZF files with chosen member cuts,
extra subfields and level-0 members."""
import struct
import zlib

import numpy as np

from tests import bam_spec

NQ = 94
EOF_BLOCK = bam_spec.EOF_BLOCK


class SpecError(ValueError):
  """Malformed input: ``kind`` is 'offset' (compressed offset of a member) or 'record' (0-based ordinal)."""

  def __init__(self, kind, where, what):
    ValueError.__init__(self, '{} {}: {}'.format(kind, where, what))
    self.kind, self.where = kind, where


# ---- BGZF ---------------------------------------------------------------------------------------------

def members(data):
  """-> [(compressed offset, inflated bytes)]; checks gzip magic, the BC subfield, CRC32 and ISIZE."""
  out, off = [], 0
  while off < len(data):
    h = data[off:off + 12]
    if len(h) < 12:
      raise SpecError('offset', off, 'truncated member')
    if h[:3] != b'\x1f\x8b\x08' or not h[3] & 4:
      raise SpecError('offset', off, 'not gzip')
    flg, xlen = h[3], struct.unpack_from('<H', h, 10)[0]
    extra = data[off + 12:off + 12 + xlen]
    if len(extra) < xlen:
      raise SpecError('offset', off, 'truncated member')
    bsize, i = None, 0
    while i + 4 <= xlen:
      slen = struct.unpack_from('<H', extra, i + 2)[0]
      if extra[i:i + 2] == b'BC' and slen == 2 and i + 6 <= xlen:
        bsize = struct.unpack_from('<H', extra, i + 4)[0] + 1
      i += 4 + slen
    if bsize is None:
      raise SpecError('offset', off, 'no BC subfield')
    m = data[off:off + bsize]
    if len(m) < bsize:
      raise SpecError('offset', off, 'truncated member')
    p = 12 + xlen
    for f in (8, 16):
      if flg & f:
        p = m.index(b'\0', p) + 1
    if flg & 2:
      p += 2
    crc, isize = struct.unpack_from('<II', m, bsize - 8)
    if isize > 65536:
      raise SpecError('offset', off, 'ISIZE')
    try:
      d = zlib.decompressobj(-15)
      raw = d.decompress(m[p:bsize - 8])
      if not d.eof or d.unused_data:
        raise zlib.error('stream does not end at the member end')
    except zlib.error:
      raise SpecError('offset', off, 'corrupt member')
    if len(raw) != isize:
      raise SpecError('offset', off, 'ISIZE')
    if zlib.crc32(raw) != crc:
      raise SpecError('offset', off, 'CRC32')
    out.append((off, raw))
    off += bsize
  return out


def has_eof_marker(data):
  return data.endswith(EOF_BLOCK)


def member(raw, level=6, extra=b'', fname=None):
  """One BGZF member of ``raw``: ``extra`` subfields go before BC; level 0 writes stored blocks."""
  c = zlib.compressobj(level, zlib.DEFLATED, -15)
  z = c.compress(raw) + c.flush()
  xfield = extra + b'BC\x02\x00'
  name = b'' if fname is None else fname + b'\0'
  bsize = 12 + len(xfield) + 2 + len(name) + len(z) + 8
  head = b'\x1f\x8b\x08' + bytes([4 | (8 if fname is not None else 0)]) + b'\0\0\0\0\0\xff' + struct.pack('<H', len(xfield) + 2)
  return head + xfield + struct.pack('<H', bsize - 1) + name + z + struct.pack('<II', zlib.crc32(raw), len(raw))


def bgzf(raw, cuts=65280, level=6, eof=True, extra=b'', empty_every=0):
  """BGZF bytes of ``raw``: ``cuts`` an int (fixed member size) or a list of the first member sizes (the rest is
  cut every 65280 bytes); ``level`` an int or a function of the member index; ``empty_every`` > 0 inserts an empty member after
  every that many members."""
  sizes, step = ([], cuts) if isinstance(cuts, int) else (list(cuts), 65280)
  rest = len(raw) - sum(sizes)
  sizes += [step] * (rest // step) + ([rest % step] if rest % step else [])
  out, at = [], 0
  for k, n in enumerate(sizes):
    out.append(member(raw[at:at + n], level(k) if callable(level) else level, extra))
    at += n
    if empty_every and k % empty_every == empty_every - 1:
      out.append(member(b'', 6, extra))
  assert at == len(raw)
  return b''.join(out) + (EOF_BLOCK if eof else b'')


# ---- BAM records ----------------------------------------------------------------------------------------

def record(name=b'r', flag=0, ref=0, pos=0, mapq=60, cigar=((4, 0),), seq=b'ACGT', qual=None, tlen=0, next_ref=-1, next_pos=-1,
           tags=b''):
  """One BAM record; ``qual`` a list of Phred values or None for a missing QUAL (0xFF bytes)."""
  l = len(seq)
  codes = [bam_spec.nt16(c) for c in seq]
  packed = bytes((codes[i] << 4 | (codes[i + 1] if i + 1 < l else 0)) for i in range(0, l, 2))
  q = b'\xff' * l if qual is None else bytes(qual)
  body = struct.pack('<iiBBHHHiiii', ref, pos, len(name) + 1, mapq, 4680, len(cigar), flag, l, next_ref, next_pos, tlen)
  body += name + b'\0' + b''.join(struct.pack('<I', n << 4 | op) for n, op in cigar) + packed + q + tags
  return struct.pack('<i', len(body)) + body


def header(contigs=(('c', 100000),), text='@HD\tVN:1.4\n'):
  return bam_spec.header_bytes(list(contigs), text=text)


def records(raw):
  """-> the record byte strings of an inflated BAM stream, after the header."""
  if raw[:4] != b'BAM\x01':
    raise SpecError('offset', 0, 'not a BAM file')
  l_text = struct.unpack_from('<i', raw, 4)[0]
  u = 8 + l_text
  nr = struct.unpack_from('<i', raw, u)[0]
  u += 4
  for _ in range(nr):
    u += 8 + struct.unpack_from('<i', raw, u)[0]
  out, k = [], 0
  while u < len(raw):
    if u + 4 > len(raw):
      raise SpecError('record', k, 'cut off')
    bs = struct.unpack_from('<i', raw, u)[0]
    if bs < 32:
      raise SpecError('record', k, 'block_size < 32')
    if u + 4 + bs > len(raw):
      raise SpecError('record', k, 'cut off')
    rec = raw[u:u + 4 + bs]
    l_name, n_cig, l_seq = rec[12], struct.unpack_from('<H', rec, 16)[0], struct.unpack_from('<i', rec, 20)[0]
    e = 32 + l_name
    if e > bs:
      raise SpecError('record', k, 'read name overruns')
    e += 4 * n_cig
    if e > bs:
      raise SpecError('record', k, 'CIGAR overruns')
    if l_seq < 0 or e + (l_seq + 1) // 2 > bs:
      raise SpecError('record', k, 'SEQ overruns')
    if e + (l_seq + 1) // 2 + l_seq > bs:
      raise SpecError('record', k, 'QUAL overruns')
    out.append(rec)
    u += 4 + bs
    k += 1
  return out


SKIPS = ('skip_flag', 'skip_mapq', 'skip_empty', 'skip_noqual', 'skip_long')


def count_records(recs, max_bp=300, max_tlen=1000, min_mq=0, every=1):
  """The counting rules over a list of record byte strings -> dict of bq_mat, len_hist, tlen and counters."""
  bq = np.zeros((2, max_bp, NQ), dtype=np.uint64)
  lh = np.zeros(max_bp + 1, dtype=np.uint64)
  tl = np.zeros(max_tlen, dtype=np.uint64)
  c = dict.fromkeys(('records', 'considered', 'counted') + SKIPS, 0)
  c['records'] = len(recs)
  for k, rec in enumerate(recs):
    if k % every:
      continue
    c['considered'] += 1
    l_name, mapq = rec[12], rec[13]
    n_cig, flag = struct.unpack_from('<HH', rec, 16)
    l_seq, tlen = struct.unpack_from('<i', rec, 20)[0], struct.unpack_from('<i', rec, 32)[0]
    qo = 36 + l_name + 4 * n_cig + (l_seq + 1) // 2
    if flag & 0xB04:
      why = 'skip_flag'
    elif mapq < min_mq:
      why = 'skip_mapq'
    elif l_seq == 0:
      why = 'skip_empty'
    elif rec[qo] == 0xFF:
      why = 'skip_noqual'
    elif l_seq > max_bp:
      why = 'skip_long'
    else:
      why = 'counted'
    c[why] += 1
    if why != 'counted':
      continue
    mate = 1 if flag & 0xC1 == 0x81 else 0
    q = np.minimum(np.frombuffer(rec, dtype=np.uint8, count=l_seq, offset=qo), NQ - 1).astype(np.int64)
    if flag & 0x10:
      q = q[::-1]
    bq[mate, np.arange(l_seq), q] += 1
    lh[l_seq] += 1
    if flag & 0xC1 == 0x41 and abs(tlen) < max_tlen:
      tl[abs(tlen)] += 1
  out = {'bq_mat': bq, 'len_hist': lh, 'tlen': tl}
  out.update(c)
  return out


def counts(data, **kw):
  """The counts of a BGZF BAM file's bytes."""
  return count_records(records(b''.join(raw for _, raw in members(data))), **kw)
