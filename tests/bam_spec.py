"""Independent pure-Python specification of the god-aligner's output (struct + zlib only): the BAM header
and records built from ``parse_qname`` + the FASTQ, a stable sort in Python, BGZF member parsing and the
BAI built from the decompressed stream and the member offsets (SAM spec v1 §4.2, §5.2, §5.3)."""
import struct
import zlib

from mitty_b200.simulation.readgenerate import parse_qname

BLOCK = 65280
NT16 = {c: i for i, c in enumerate('=ACMGRSVTWYHKDBN')}
CIGAR_OPS = {'=': 7, 'X': 8, 'I': 1, 'D': 2}
EOF_BLOCK = bytes.fromhex('1f8b08040000000000ff0600424302001b0003000000000000000000')


def nt16(c):
  return NT16.get(chr(c).upper(), 15) if chr(c) != '=' else 0


def nt16_comp(x):
  return (x & 1) << 3 | (x & 2) << 1 | (x & 4) >> 1 | (x & 8) >> 3


def reg2bin(beg, end):
  end -= 1
  for shift, first in ((14, 4681), (17, 585), (20, 73), (23, 9), (26, 1)):
    if beg >> shift == end >> shift:
      return first + (beg >> shift)
  return 0


def reg2bins(beg, end):
  """Bins that may hold records overlapping [beg, end) (SAM spec §5.3)."""
  end -= 1
  out = [0]
  for shift, first in ((26, 1), (23, 9), (20, 73), (17, 585), (14, 4681)):
    out += range(first + (beg >> shift), first + (end >> shift) + 1)
  return out


def cigar_ops(cigar):
  """'150=' / '13=8I129=' -> [(n, op)]; the plain CIGAR of parse_qname ('>p:nI' is already 'nI')."""
  import re
  ops = re.findall(r'(\d+)(\D)', cigar)
  assert ''.join(n + o for n, o in ops) == cigar, cigar
  return [(int(n), o) for n, o in ops]


def span(cigar):
  return sum(n for n, o in cigar_ops(cigar) if o in '=XD')


def end_of(pos0, cigar):
  return pos0 + max(span(cigar), 1)


def header_text(contigs, sample):
  return ('@HD\tVN:1.4\tSO:coordinate\n' + ''.join('@SQ\tSN:{}\tLN:{}\n'.format(n, l) for n, l in contigs) +
          '@RG\tID:{0}\tSM:{0}\tPL:ILLUMINA\n'.format(sample))


def header_bytes(contigs, sample=None, text=None):
  text = (header_text(contigs, sample) if text is None else text).encode()
  h = b'BAM\x01' + struct.pack('<i', len(text)) + text + struct.pack('<i', len(contigs))
  for n, l in contigs:
    h += struct.pack('<i', len(n) + 1) + n.encode() + b'\0' + struct.pack('<i', l)
  return h


def encode_record(name, seq, qual, info, mate, file_index, ref_id, sample):
  """One BAM record: info / mate = parse_qname's ReadInfo of this read and of its mate (None: single-end)."""
  pos = info.pos - 1
  end = end_of(pos, info.cigar)
  flag = 0x10 if info.strand else 0
  next_ref, next_pos, tlen = -1, -1, 0
  if mate is not None:
    flag |= 0x1 | 0x2 | (0x80 if file_index else 0x40) | (0x20 if mate.strand else 0)
    mpos = mate.pos - 1
    mend = end_of(mpos, mate.cigar)
    next_ref, next_pos = ref_id, mpos
    lo, hi = min(pos, mpos), max(end, mend)
    tlen = hi - lo if (pos < mpos or (pos == mpos and file_index == 0)) else lo - hi
  codes = [nt16(c) for c in seq]
  q = [c - 33 for c in qual]
  if info.strand:
    codes = [nt16_comp(c) for c in reversed(codes)]
    q = q[::-1]
  packed = bytes((codes[i] << 4 | (codes[i + 1] if i + 1 < len(codes) else 0)) for i in range(0, len(codes), 2))
  ops = cigar_ops(info.cigar)
  body = struct.pack('<iiBBHHHiiii', ref_id, pos, len(name) + 1, 60, reg2bin(pos, end), len(ops), flag, len(seq), next_ref, next_pos, tlen)
  body += name + b'\0' + b''.join(struct.pack('<I', n << 4 | CIGAR_OPS[o]) for n, o in ops) + packed + bytes(x & 0xFF for x in q)
  body += b'RGZ' + sample.encode() + b'\0'
  return struct.pack('<i', len(body)) + body


def fastq_records(buf):
  lines = buf.split(b'\n')
  return [(lines[k][1:], lines[k + 1], lines[k + 3]) for k in range(0, len(lines) - 3, 4)]


def records(contigs, fq1, fq2=None):
  """-> the sorted records (list of bytes): one per read, stable sort on (refID, pos, reverse bit)."""
  ref_ids = {n: i for i, (n, _) in enumerate(contigs)}
  files = [fastq_records(fq1)] + ([fastq_records(fq2)] if fq2 is not None else [])
  n = min(len(f) for f in files)
  sample = files[0][0][0].decode().split('|', 1)[0].split(':', 1)[0] if n else ''
  out = []
  for t in range(n):
    for f, recs in enumerate(files):
      name, seq, qual = recs[t]
      infos = parse_qname(name.decode())
      info = infos[f]
      mate = infos[1 - f] if fq2 is not None else None
      rid = ref_ids[info.chrom]
      assert info.pos - 1 >= 0 and info.pos - 1 + span(info.cigar) <= contigs[rid][1]
      out.append(((rid, info.pos - 1, info.strand), len(out), encode_record(name, seq, qual, info, mate, f, rid, sample)))
  out.sort(key=lambda r: (r[0], r[1]))
  return sample, [r[2] for r in out]


def bam_bytes(contigs, fq1, fq2=None):
  """The uncompressed BAM stream the god-aligner must write."""
  sample, recs = records(contigs, fq1, fq2)
  return header_bytes(contigs, sample) + b''.join(recs)


# ---- BGZF ---------------------------------------------------------------------------------------------

def members(data):
  """-> [(compressed offset, decompressed bytes)] of a BGZF file; checks the framing of every member."""
  out, off = [], 0
  while off < len(data):
    assert data[off:off + 4] == b'\x1f\x8b\x08\x04', off
    xlen = struct.unpack_from('<H', data, off + 10)[0]
    assert xlen == 6 and data[off + 12:off + 16] == b'BC\x02\x00'
    bsize = struct.unpack_from('<H', data, off + 16)[0] + 1
    assert bsize <= 65536
    member = data[off:off + bsize]
    raw = zlib.decompress(member[18:-8], -15)
    crc, isize = struct.unpack_from('<II', member, bsize - 8)
    assert crc == zlib.crc32(raw) and isize == len(raw)
    out.append((off, raw))
    off += bsize
  return out


def decompress(data):
  return b''.join(raw for _, raw in members(data))


# ---- BAI ----------------------------------------------------------------------------------------------

def build_bai(data, n_ref):
  """The index of a BGZF BAM file, built from its decompressed stream and member offsets: consecutive
  records of one bin form one chunk; linear index = first record overlapping each 16 kb window (empty
  windows take the next window's value); pseudo-bin 37450 per reference; n_no_coor = 0."""
  ms = members(data)
  starts = [off for off, _ in ms]
  sizes = [len(raw) for _, raw in ms]
  # fixed cuts: every member but the last data one and the EOF member holds BLOCK bytes
  assert all(s == BLOCK for s in sizes[:-2]) and sizes[-1] == 0 and data[-28:] == EOF_BLOCK

  def v(u):
    return starts[u // BLOCK] << 16 | u % BLOCK

  raw = b''.join(r for _, r in ms)
  l_text = struct.unpack_from('<i', raw, 4)[0]
  u = 8 + l_text
  nr = struct.unpack_from('<i', raw, u)[0]
  u += 4
  for _ in range(nr):
    ln = struct.unpack_from('<i', raw, u)[0]
    u += 8 + ln
  refs = [{'bins': {}, 'lin': [], 'beg': 0, 'end': 0, 'n': 0} for _ in range(n_ref)]
  cur = None
  while u < len(raw):
    bs = struct.unpack_from('<i', raw, u)[0]
    ref, pos, bmn, fnc = struct.unpack_from('<iiII', raw, u + 4)
    l_name, n_cig, b = bmn & 0xFF, fnc & 0xFFFF, bmn >> 16
    cig = struct.unpack_from('<{}I'.format(n_cig), raw, u + 36 + l_name)
    sp = sum(c >> 4 for c in cig if (c & 15) in (0, 2, 3, 7, 8))
    end = pos + max(sp, 1)
    ub, ue = u, u + 4 + bs
    if cur is None or cur[0] != ref or cur[1] != b:
      cur = [ref, b, ub, ue]
      refs[ref]['bins'].setdefault(b, []).append(cur)
    cur[3] = ue
    R = refs[ref]
    if R['n'] == 0:
      R['beg'] = ub
    R['end'] = ue
    R['n'] += 1
    lin = R['lin']
    if len(lin) <= (end - 1) >> 14:
      lin += [None] * (((end - 1) >> 14) + 1 - len(lin))
    for w in range(pos >> 14, ((end - 1) >> 14) + 1):
      if lin[w] is None:
        lin[w] = ub
    u = ue
  out = b'BAI\x01' + struct.pack('<i', n_ref)
  for R in refs:
    out += struct.pack('<i', len(R['bins']) + (1 if R['n'] else 0))
    for b in sorted(R['bins']):
      out += struct.pack('<Ii', b, len(R['bins'][b])) + b''.join(struct.pack('<QQ', v(c[2]), v(c[3])) for c in R['bins'][b])
    if R['n']:
      out += struct.pack('<Ii', 37450, 2) + struct.pack('<QQQQ', v(R['beg']), v(R['end']), R['n'], 0)
    lin = R['lin']
    for w in range(len(lin) - 2, -1, -1):
      if lin[w] is None:
        lin[w] = lin[w + 1]
    out += struct.pack('<i', len(lin)) + b''.join(struct.pack('<Q', v(x)) for x in lin)
  return out + struct.pack('<Q', 0)


def parse_bai(bai):
  """-> [ {bin: [(beg, end)]}, [linear offsets] ] per reference."""
  assert bai[:4] == b'BAI\x01'
  n_ref = struct.unpack_from('<i', bai, 4)[0]
  off, out = 8, []
  for _ in range(n_ref):
    n_bin = struct.unpack_from('<i', bai, off)[0]
    off += 4
    bins = {}
    for _ in range(n_bin):
      b, nc = struct.unpack_from('<Ii', bai, off)
      off += 8
      bins[b] = [struct.unpack_from('<QQ', bai, off + 16 * i) for i in range(nc)]
      off += 16 * nc
    n_intv = struct.unpack_from('<i', bai, off)[0]
    lin = list(struct.unpack_from('<{}Q'.format(n_intv), bai, off + 4))
    off += 4 + 8 * n_intv
    out.append((bins, lin))
  return out


def query(index, ref, beg, end):
  """Chunks (virtual offsets) the index returns for [beg, end) of reference ``ref``."""
  bins, lin = index[ref]
  w = beg >> 14
  min_off = lin[w] if w < len(lin) else (lin[-1] if lin else 0)
  return [(a, b) for bn in reg2bins(beg, end) if bn in bins and bn != 37450 for a, b in bins[bn] if b > min_off]


def record_offsets(data):
  """-> [(virtual offset, refID, pos, end)] of every record of a BGZF BAM file."""
  ms = members(data)
  starts = [off for off, _ in ms]
  raw = b''.join(r for _, r in ms)
  l_text = struct.unpack_from('<i', raw, 4)[0]
  u = 8 + l_text
  nr = struct.unpack_from('<i', raw, u)[0]
  u += 4
  for _ in range(nr):
    u += 8 + struct.unpack_from('<i', raw, u)[0]
  out = []
  while u < len(raw):
    bs, ref, pos, bmn, fnc = struct.unpack_from('<iiiII', raw, u)
    cig = struct.unpack_from('<{}I'.format(fnc & 0xFFFF), raw, u + 36 + (bmn & 0xFF))
    sp = sum(c >> 4 for c in cig if (c & 15) in (0, 2, 3, 7, 8))
    out.append((starts[u // BLOCK] << 16 | u % BLOCK, ref, pos, pos + max(sp, 1)))
    u += 4 + bs
  return out


def decode_reads(raw):
  """BAM stream -> [(qname, flag, seq, qual)] with strand-1 reads turned back into their FASTQ form."""
  l_text = struct.unpack_from('<i', raw, 4)[0]
  u = 8 + l_text
  nr = struct.unpack_from('<i', raw, u)[0]
  u += 4
  for _ in range(nr):
    u += 8 + struct.unpack_from('<i', raw, u)[0]
  out = []
  while u < len(raw):
    bs, ref, pos, bmn, fnc, l_seq = struct.unpack_from('<iiiIIi', raw, u)
    l_name, n_cig, flag = bmn & 0xFF, fnc & 0xFFFF, fnc >> 16
    p = u + 36
    name = raw[p:p + l_name - 1]
    p += l_name + 4 * n_cig
    codes = [(raw[p + i // 2] >> (4 if i % 2 == 0 else 0)) & 15 for i in range(l_seq)]
    p += (l_seq + 1) // 2
    qual = [x + 33 for x in raw[p:p + l_seq]]
    if flag & 0x10:
      codes = [nt16_comp(c) for c in reversed(codes)]
      qual = qual[::-1]
    out.append((name, flag, bytes(ord('=ACMGRSVTWYHKDBN'[c]) for c in codes), bytes(qual)))
    u += 4 + bs
  return out
