"""Numpy restatement of the engine's PRODUCTION-mode corruption (the draw layout documented at
MgCorruptCtx in mitty_b200/csrc/mg_core.cuh): one Philox4x32-7 block per four cycles, one 32-bit
word and one lookup in a Vose alias row over the joint outcomes (quality, substitution) per base.
Test infrastructure: lets the fused GPU path and the standalone corrupt kernel be checked byte for
byte, not only statistically."""
import re

import numpy as np

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = 0x9E3779B9, 0xBB67AE85
STREAM_CORRUPT = 0x636f7272
CORRUPT_ROUNDS = 7   # MG_CORRUPT_ROUNDS: the per-base corruption stream is Philox4x32-7
MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
  return philox4x32(c0, c1, c2, c3, k0, k1, 10)


def philox4x32(c0, c1, c2, c3, k0, k1, rounds=10):
  c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) & MASK for c in (c0, c1, c2, c3))
  k0, k1 = int(k0) & 0xFFFFFFFF, int(k1) & 0xFFFFFFFF
  for _ in range(rounds):
    p0, p1 = M0 * c0, M1 * c2
    h0, l0, h1, l1 = p0 >> np.uint64(32), p0 & MASK, p1 >> np.uint64(32), p1 & MASK
    c0, c1, c2, c3 = h1 ^ c1 ^ np.uint64(k0), l1, h0 ^ c3 ^ np.uint64(k1), l0
    k0, k1 = (k0 + W0) & 0xFFFFFFFF, (k1 + W1) & 0xFFFFFFFF
  return [c.astype(np.uint32) for c in (c0, c1, c2, c3)]


def quality_masses(row, clip=93):
  """Outcome probabilities of searchsorted(row, u, side='left') clipped to `clip`, u uniform in [0,1)
  (illumina.py:156) -- ss_left_probs in mg_api.cu, same operation order."""
  n_bq = len(row)
  q = [0.0] * (clip + 1)
  prev = 0.0
  for b in range(n_bq):
    c = min(float(row[b]), 1.0)
    if c < prev:
      c = prev
    q[min(b, clip)] += c - prev
    prev = c
  q[min(n_bq, clip)] += 1.0 - prev
  return q


def row_outcomes(row, phred_p, code9):
  """[(code, mass)] of the outcomes with non-zero mass of one (mate, cycle): (q, 0) "called
  correctly" with P(q)(1 - phred_p[q]) and (q, s), s = 1..3, with P(q) phred_p[q] / 3 each
  (build_joint_row in mg_api.cu, same order).  code = s << 6 | q, or s << 7 | q with 9-bit codes."""
  qb = 7 if code9 else 6
  out = []
  for b, pq in enumerate(quality_masses(row)):
    if pq <= 0.0:
      continue
    p = float(phred_p[b]) if b < 100 else 0.0
    m0, m = pq * (1.0 - p), pq * p / 3.0
    if m0 > 0.0:
      out.append((b, m0))
    if m > 0.0:
      out += [((1 << qb) | b, m), ((2 << qb) | b, m), ((3 << qb) | b, m)]
  return out


def table_shape(cum_bq_mat, phred_p, n_rows):
  """(kshift, code9) the library picks for the first n_rows cycles: 9-bit codes iff some quality >= 64
  carries mass, K = 2^kshift = the smallest power of two (>= 32) that holds the longest outcome list."""
  m = np.asarray(cum_bq_mat, dtype=np.float64)
  code9, longest = 0, 1
  for mi in range(m.shape[0]):
    for ci in range(min(n_rows, m.shape[1])):
      qm = quality_masses(m[mi, ci])
      if any(v > 0.0 for v in qm[64:]):
        code9 = 1
      longest = max(longest, len(row_outcomes(m[mi, ci], phred_p, 1)))
  ks = 5
  while (1 << ks) < longest:
    ks += 1
  return ks, code9


def _vose(q, K):
  """Vose's alias method, the same operation order as vose() in mg_api.cu -> (prob[K], alias[K])."""
  q = list(q)
  small, large = [], []
  for i in range(K):
    q[i] *= K
    (small if q[i] < 1.0 else large).append(i)
  prob, alias = [1.0] * K, list(range(K))
  while small and large:
    s, l = small.pop(), large.pop()
    prob[s], alias[s] = q[s], l
    q[l] = (q[l] + q[s]) - 1.0
    (small if q[l] < 1.0 else large).append(l)
  return prob, alias


def joint_tables(cum_bq_mat, phred_p, kshift, code9, n_rows=None):
  """-> alias u32[n_mates, n_cycles, 1 << kshift]: per (mate, cycle) the Vose alias row over that
  cycle's outcome list; entry = thr << (32 - tb) | self code << cb | alias code with (tb, cb) = (16, 8)
  or (14, 9).  Entries beyond the list have threshold 0 and both codes = their alias' code; an entry
  whose threshold rounds to 0 (to the maximum) carries its alias' (its own) code in both fields.
  Only the first n_rows cycles are built (the rest stay zero)."""
  m = np.asarray(cum_bq_mat, dtype=np.float64)
  n_mates, n_cycles, _ = m.shape
  K = 1 << kshift
  tb, cb = (14, 9) if code9 else (16, 8)
  out = np.zeros((n_mates, n_cycles, K), dtype=np.uint32)
  for mi in range(n_mates):
    for ci in range(n_cycles if n_rows is None else min(n_rows, n_cycles)):
      oc = row_outcomes(m[mi, ci], phred_p, code9)
      assert 0 < len(oc) <= K
      tot = 0.0
      for _, v in oc:
        tot += v
      q = [v / tot for _, v in oc] + [0.0] * (K - len(oc))
      prob, alias = _vose(q, K)
      for i in range(K):
        pr = min(max(prob[i], 0.0), 1.0)
        t = min(int(np.floor(pr * float(1 << tb) + 0.5)), (1 << tb) - 1)
        a = oc[alias[i]][0] if alias[i] < len(oc) else oc[0][0]
        s = oc[i][0] if i < len(oc) else a
        if t == 0:
          s = a
        if t == (1 << tb) - 1:
          a = s
        out[mi, ci, i] = (t << (32 - tb)) | (s << cb) | a
  return out


def row_distribution(alias_row, kshift, code9):
  """{code: probability} encoded by one alias row (exact rational arithmetic on the 32-bit entries:
  take iff w < e, w uniform)."""
  K = 1 << kshift
  cb = 9 if code9 else 8
  p = {}
  for i in range(K):
    e = int(alias_row[i])
    take = e / 4294967296.0
    s, a = (e >> cb) & ((1 << cb) - 1), e & ((1 << cb) - 1)
    p[s] = p.get(s, 0.0) + take / K
    p[a] = p.get(a, 0.0) + (1.0 - take) / K
  return p


def fused_tables(eng, which=0):
  """The tables the library built at load time (which = 0: the emit kernel's, cycles < rlen; 1: the
  standalone corrupt kernel's, every cycle) -> (alias, kshift, code9)."""
  return eng.model_tables(which)


BASES = b'ACGT'
CODE = {65: 0, 67: 1, 71: 2, 84: 3}


def record_name(header):
  """FastxFile's .name of a header line: the bytes after its first one, up to the first space, tab or CR."""
  return re.split(b'[ \t\r]', header[1:], maxsplit=1)[0]


def corrupt_file(fq, f, tables, k0, k1, serials=None, names_from=None):
  """Corrupt a perfect FASTQ buffer (file index f) -> bytes.  tables = (alias, kshift, code9).
  serials: per-record template serial (default 0..n-1, the standalone kernel's numbering).
  names_from: FASTQ buffer whose record names head the output records, '@' + record_name() -- the
  standalone corrupt-reads writes read 1's name on both files (readcorrupt.py:113); default: every
  record keeps its own header line, as the fused emit kernel does."""
  alias, kshift, code9 = tables
  qb = 7 if code9 else 6
  cb = 9 if code9 else 8
  lines = fq.split(b'\n')
  n_rec = (len(lines) - 1) // 4
  if serials is None:
    serials = np.arange(n_rec, dtype=np.uint64)
  heads = [lines[4 * rec] for rec in range(n_rec)]
  if names_from is not None:
    src = names_from.split(b'\n')
    heads = [b'@' + record_name(src[4 * rec]) for rec in range(n_rec)]
  out = []
  L = max(len(lines[4 * r + 1]) for r in range(n_rec)) if n_rec else 0
  ng = (L + 3) // 4
  s_grid = np.repeat(np.asarray(serials, dtype=np.uint64), ng)
  g_grid = np.tile(np.arange(ng, dtype=np.uint64), n_rec)
  r = philox4x32(s_grid & MASK, (s_grid >> np.uint64(32)) * np.uint64(2) + np.uint64(f), g_grid, STREAM_CORRUPT, k0, k1, CORRUPT_ROUNDS)
  w_all = np.stack(r, axis=1).reshape(n_rec, ng * 4)
  n_cycles = alias.shape[1]
  flat = alias[f].reshape(-1).astype(np.uint64)
  for rec in range(n_rec):
    seq = bytearray(lines[4 * rec + 1])
    Lr = len(seq)
    w = w_all[rec, :Lr].astype(np.uint64)
    idx = (w & np.uint64((1 << kshift) - 1)).astype(np.int64)          # the entry: w's low bits
    e = flat[(np.arange(Lr, dtype=np.int64) << kshift) | idx]
    take = w < e                                                       # the threshold sits in e's top bits: w's high bits decide
    code = np.where(take, e >> np.uint64(cb), e) & np.uint64((1 << cb) - 1)
    q = (code & np.uint64((1 << qb) - 1)).astype(np.int64)
    s = (code >> np.uint64(qb)).astype(np.int64)
    for n in np.flatnonzero(s):
      c = CODE.get(seq[n])
      seq[n] = ord('N') if c is None else BASES[c ^ int(s[n])]
    out.append(heads[rec] + b'\n' + bytes(seq) + b'\n+\n' + (q + 33).astype(np.uint8).tobytes() + b'\n')
  return b''.join(out)
