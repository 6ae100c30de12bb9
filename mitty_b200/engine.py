"""Host-side handle on one GPU: a thin, typed layer over the C ABI (include/mitty_b200.h).

One ``Engine`` = one ``mg_ctx`` = one GPU + one CUDA stream.  Everything numeric happens in the
CUDA library; this module only moves numpy buffers across the boundary and turns status codes into
the exceptions the reference raises (ValueError / IndexError).
"""
import ctypes as C

import numpy as np

from mitty_b200 import _lib
from mitty_b200._lib import MODE_DET, MODE_EXPLICIT, MODE_PHILOX, UnitDesc

SEED_MAX = (1 << 32) - 1  # illumina.py:9
PHRED_P = 10 ** (-np.arange(100) / 10)  # illumina.py:137


def _ptr(a):
  return None if a is None else C.c_void_p(a.ctypes.data)


def _u8(buf):
  return buf if buf is None or isinstance(buf, np.ndarray) else np.frombuffer(buf, dtype=np.uint8)


def _fastq_args(fq1, fq2):
  """FASTQ buffers 1 and 2 (bytes or uint8 arrays; fq2 may be None) as the C ABI's (pointer, length) pairs; an
  empty buffer 1 is passed as a non-null address, which the library does not read."""
  a1, a2 = _u8(fq1), _u8(fq2)
  return _ptr(a1 if a1.size else np.zeros(1, np.uint8)), a1.size, _ptr(a2), 0 if a2 is None else a2.size


class CopyHandle(object):
  __slots__ = ('id', 'p_min', 'p_max', 'n_nodes', 'region')

  def __init__(self, id_, p_min, p_max, n_nodes, region):
    self.id, self.p_min, self.p_max, self.n_nodes, self.region = id_, p_min, p_max, n_nodes, region


class BatchHandle(object):
  """Many small (region, copy) segments built as one node table / haplotype (mg_batch_build)."""
  __slots__ = ('id', 'p_min', 'p_max', 'n_segs')

  def __init__(self, id_, p_min, p_max):
    self.id, self.p_min, self.p_max, self.n_segs = id_, p_min, p_max, len(p_min)


BATCH_MAX_CANDIDATES = 2048   # MG_BATCH_MAXC: candidates per unit on the batch path


class Engine(object):
  def __init__(self, device=0, stream=None):
    self._L = _lib.lib()
    h = C.c_void_p()
    rc = self._L.mg_ctx_create(int(device), C.c_void_p(stream) if stream else None, C.byref(h))
    if rc != 0:
      raise RuntimeError('mitty_b200: cannot create a context on CUDA device {} (rc={}); the engine has no CPU fallback'.format(device, rc))
    self._h = h
    self.device = device
    self.rlen = None
    self._keep = []
    self._pinned = []

  def close(self):
    if getattr(self, '_h', None):
      for p in self._pinned:
        self._L.mg_host_free(self._h, p)
      self._pinned = []
      self._L.mg_ctx_destroy(self._h)
      self._h = None

  def __del__(self):
    try:
      self.close()
    except Exception:
      pass

  def _check(self, rc):
    if rc == 0:
      return
    msg = self._L.mg_last_error(self._h).decode()
    if rc == _lib.MG_EVALUE:
      raise ValueError(msg)
    if rc == _lib.MG_EINDEX:
      raise IndexError(msg)
    if rc == _lib.MG_ECAP:
      raise BufferError(msg)
    raise RuntimeError('mitty_b200 rc={}: {}'.format(rc, msg))

  def synchronize(self):
    self._check(self._L.mg_synchronize(self._h))

  # -- pinned host buffers ----------------------------------------------------------------------
  def pinned(self, nbytes):
    """uint8 numpy array over page-locked host memory (freed with the engine)."""
    p = C.c_void_p()
    self._check(self._L.mg_host_alloc(self._h, int(nbytes), C.byref(p)))
    self._pinned.append(p)
    buf = (C.c_uint8 * int(nbytes)).from_address(p.value)
    return np.frombuffer(buf, dtype=np.uint8)

  # -- model -------------------------------------------------------------------------------------
  def load_model(self, model, rlen=None):
    """model: dict with cum_tlen, cum_bq_mat (raw .pkl model or read_model_params output)."""
    cum_tlen = np.ascontiguousarray(model['cum_tlen'], dtype=np.float64)
    cum_bq = np.ascontiguousarray(model['cum_bq_mat'], dtype=np.float64)
    if rlen is None:
      rlen = model['rlen'] if 'rlen' in model else model['mean_rlen']
    self.rlen = int(rlen)
    self._model_shape = cum_bq.shape
    self._check(self._L.mg_model_load(self._h, _ptr(cum_tlen), cum_tlen.size, _ptr(cum_bq), cum_bq.shape[0],
                                      cum_bq.shape[1], cum_bq.shape[2], _ptr(PHRED_P), self.rlen))

  def model_tables(self, which=0):
    """-> (alias u32[n_mates, n_cycles, 1 << kshift], kshift, code9) as built at load time: the joint
    (quality, substitution) alias rows of production-mode corruption.  which = 0: the fused emit kernel's
    table (cycles < rlen), 1: the standalone corrupt kernel's (every cycle)."""
    ks, c9, nr = C.c_int32(0), C.c_int32(0), C.c_int32(0)
    self._check(self._L.mg_model_tables(self._h, int(which), None, 0, C.byref(ks), C.byref(c9), C.byref(nr)))
    nm, nc = self._model_shape[0], self._model_shape[1]
    alias = np.zeros((nm * nc) << ks.value, dtype=np.uint32)
    self._check(self._L.mg_model_tables(self._h, int(which), _ptr(alias), alias.size, C.byref(ks), C.byref(c9), C.byref(nr)))
    return alias.reshape(nm, nc, 1 << ks.value), ks.value, c9.value

  # -- bam2illumina -----------------------------------------------------------------------------
  def read_model_counts(self, path, max_bp=300, max_tlen=1000, min_mq=0, every=1, threads=1, chunk_bytes=64 << 20):
    """mg_readmodel_bam: the per-base counts of an Illumina read model over a BGZF BAM (file or FIFO).
    -> dict with bq_mat u64[2, max_bp, 94], len_hist u64[max_bp + 1], tlen u64[max_tlen], the counters of
    READ_MODEL_COUNTS, 'times' (ms: read, inflate, walk, h2d, kernel, total) and 'thread_ms' (busy time of each
    inflate thread).  Malformed input raises ValueError naming the record ordinal or compressed offset."""
    threads = max(1, int(threads))
    bq = np.zeros((2, int(max_bp), 94), dtype=np.uint64)
    lh = np.zeros(int(max_bp) + 1, dtype=np.uint64)
    tl = np.zeros(int(max_tlen), dtype=np.uint64)
    cnt, times, tms = np.zeros(12, dtype=np.int64), np.zeros(6, dtype=np.float64), np.zeros(threads, dtype=np.float64)
    bw, bc = C.c_int64(-1), C.c_int32(0)
    rc = self._L.mg_readmodel_bam(self._h, str(path).encode(), int(max_bp), int(max_tlen), int(min_mq), int(every), threads, int(chunk_bytes),
                                  _ptr(bq), _ptr(lh), _ptr(tl), _ptr(cnt), _ptr(times), _ptr(tms), C.byref(bw), C.byref(bc))
    if rc == _lib.MG_EVALUE and bc.value:
      raise bam_read_error(path, bc.value, bw.value)
    self._check(rc)
    out = {'bq_mat': bq, 'len_hist': lh, 'tlen': tl, 'thread_ms': tms,
           'times': dict(zip(('read_ms', 'inflate_ms', 'walk_ms', 'h2d_ms', 'kernel_ms', 'total_ms'), (float(x) for x in times)))}
    out.update(zip(READ_MODEL_COUNTS, (int(x) for x in cnt)))
    return out

  # -- alignment-analysis -----------------------------------------------------------------------
  def alignment_error_counts(self, path, max_d=200, max_size=50, threads=1, chunk_bytes=64 << 20):
    """mg_alnerr_bam: an aligner's BAM (file or FIFO) scored against the truth in the qnames.  -> dict with
    mq u64[256, 2 * max_d + 3] (rows MAPQ, columns d_err -max_d .. max_d, wrong chrom, unmapped), vsize
    u64[2 * max_size + 4, 2 * max_d + 3] (rows variant size < -max_size, -max_size .. max_size, > max_size, no
    variant), the counters of ALIGNMENT_COUNTS, 'times' (ms: read, inflate, walk, h2d, kernel, total) and
    'thread_ms'.  Malformed input raises ValueError naming the record ordinal or compressed offset."""
    threads, max_d, max_size = max(1, int(threads)), int(max_d), int(max_size)
    mq = np.zeros((256, 2 * max_d + 3), dtype=np.uint64)
    vs = np.zeros((2 * max_size + 4, 2 * max_d + 3), dtype=np.uint64)
    cnt, times, tms = np.zeros(len(ALIGNMENT_COUNTS), dtype=np.int64), np.zeros(6, dtype=np.float64), np.zeros(threads, dtype=np.float64)
    bw, bc = C.c_int64(-1), C.c_int32(0)
    rc = self._L.mg_alnerr_bam(self._h, str(path).encode(), max_d, max_size, threads, int(chunk_bytes), _ptr(mq), _ptr(vs), _ptr(cnt), _ptr(times),
                               _ptr(tms), C.byref(bw), C.byref(bc))
    if rc == _lib.MG_EVALUE and bc.value:
      raise bam_read_error(path, bc.value, bw.value)
    self._check(rc)
    out = {'mq': mq, 'vsize': vs, 'thread_ms': tms,
           'times': dict(zip(('read_ms', 'inflate_ms', 'walk_ms', 'h2d_ms', 'kernel_ms', 'total_ms'), (float(x) for x in times)))}
    out.update(zip(ALIGNMENT_COUNTS, (int(x) for x in cnt)))
    return out

  # -- haplotypes --------------------------------------------------------------------------------
  def load_region(self, ref_bytes, bed_start):
    ref = np.ascontiguousarray(ref_bytes, dtype=np.uint8)
    rid = C.c_int64(0)
    self._check(self._L.mg_region_load(self._h, _ptr(ref) if ref.size else None, ref.size, int(bed_start), C.byref(rid)))
    return rid.value

  def free_region(self, rid):
    self._check(self._L.mg_region_free(self._h, rid))

  def build_copy(self, rid, vl):
    """vl: mitty_b200.lib.vcfio.VariantList of the variants on this chromosome copy."""
    cid, p_min, p_max, nn = C.c_int64(0), C.c_int64(0), C.c_int64(0), C.c_int64(0)
    n = len(vl)
    alt_pool = vl.alt_pool if vl.alt_pool.size else np.zeros(1, dtype=np.uint8)
    self._check(self._L.mg_copy_build(self._h, rid, n, _ptr(vl.pos), _ptr(vl.op), _ptr(vl.oplen), _ptr(alt_pool),
                                      _ptr(vl.alt_off), C.byref(cid), C.byref(p_min), C.byref(p_max), C.byref(nn)))
    return CopyHandle(cid.value, p_min.value, p_max.value, nn.value, rid)

  def free_copy(self, cp):
    self._check(self._L.mg_copy_free(self._h, cp.id))

  def copy_nodes(self, cp):
    """-> (ps, pr, op, oplen) arrays: the reference's Node fields (rpc.py:5-35)."""
    n = cp.n_nodes
    ps, pr, oplen = (np.empty(n, dtype=np.int64) for _ in range(3))
    op = np.empty(n, dtype=np.uint8)
    self._check(self._L.mg_copy_nodes(self._h, cp.id, _ptr(ps), _ptr(pr), _ptr(op), _ptr(oplen)))
    return ps, pr, op, oplen

  def copy_haplotype(self, cp):
    out = np.empty(max(1, cp.p_max - cp.p_min), dtype=np.uint8)
    self._check(self._L.mg_copy_haplotype(self._h, cp.id, _ptr(out), out.size))
    return out[:cp.p_max - cp.p_min]

  # -- units -------------------------------------------------------------------------------------
  def _desc(self, cp, n, p, mode, seed, ts, u_tlen, tl, fo, prefix, mid, corrupt, corrupt_seed, p_min=0, p_max=0):
    d = UnitDesc()
    d.copy_id = cp.id if cp is not None else 0
    d.n_candidates = int(n); d.p = float(p); d.mode = int(mode); d.unit_seed = int(seed) & 0xFFFFFFFF
    keep = []
    for name, a, dt in (('ts', ts, np.int64), ('u_tlen', u_tlen, np.float64), ('tl', tl, np.int64), ('fo', fo, np.int8)):
      if a is not None:
        a = np.ascontiguousarray(a, dtype=dt)
        if a.size < n:
          raise ValueError('{} has {} entries, {} candidates'.format(name, a.size, n))
        keep.append(a)
        setattr(d, name, a.ctypes.data)
    d.qname_prefix = prefix.encode() if prefix is not None else None
    d.qname_mid = mid.encode() if mid is not None else None
    d.corrupt = int(bool(corrupt)); d.corrupt_seed = int(corrupt_seed) & 0xFFFFFFFF
    d.p_min, d.p_max = int(p_min), int(p_max)
    return d, keep

  def sample_templates(self, n, p, mode, seed, cp=None, p_min=0, p_max=0, ts=None, u_tlen=None, tl=None):
    """-> per-candidate (ts, te, fo); te == -1 where te >= p_max (illumina.py:66-76)."""
    d, keep = self._desc(cp, n, p, mode, seed, ts, u_tlen, tl, None, None, None, 0, 0, p_min, p_max)
    ts_o, te_o = np.empty(max(1, n), dtype=np.int64), np.empty(max(1, n), dtype=np.int64)
    fo_o = np.empty(max(1, n), dtype=np.int8)
    self._check(self._L.mg_sample_templates(self._h, C.byref(d), _ptr(ts_o), _ptr(te_o), _ptr(fo_o)))
    return ts_o[:n], te_o[:n], fo_o[:n]

  def generate_unit(self, cp, n, p, mode, seed, prefix, mid, ts=None, u_tlen=None, tl=None, fo=None,
                    corrupt=False, corrupt_seed=0, out=None, fetch=True, wait=True):
    """One work unit -> (fastq1, fastq2, n_templates, n_te_kept, bytes per file); the two arrays are None with
    fetch=False (the unit stays on the device for ``drain_async`` / ``unit_read``).

    out: optional pair of preallocated uint8 arrays (e.g. pinned) to receive the bytes; the
    returned arrays are views of them.  fetch=False leaves the result on the device.
    wait=False (needs pinned ``out``) returns once the device-to-host copies are enqueued: the next
    unit's kernels overlap with them and the bytes are valid after ``wait_copies()``.
    """
    d, keep = self._desc(cp, n, p, mode, seed, ts, u_tlen, tl, fo, prefix, mid, corrupt, corrupt_seed)
    nb, nt, nk = C.c_int64(0), C.c_int64(0), C.c_int64(0)
    if not fetch:
      self._check(self._L.mg_unit_generate(self._h, C.byref(d), None, None, 0, C.byref(nb), C.byref(nt), C.byref(nk)))
      return None, None, nt.value, nk.value, nb.value
    if out is None:
      est = int(n) * (2 * self.rlen + 120 + len(prefix) + len(mid)) // 1 + 4096
      out = (np.empty(est, dtype=np.uint8), np.empty(est, dtype=np.uint8))
    o1, o2 = out
    gen = self._L.mg_unit_generate if wait else self._L.mg_unit_generate_async
    rc = gen(self._h, C.byref(d), _ptr(o1), _ptr(o2), min(o1.size, o2.size), C.byref(nb), C.byref(nt), C.byref(nk))
    if rc == _lib.MG_ECAP:
      o1, o2 = np.empty(nb.value, dtype=np.uint8), np.empty(nb.value, dtype=np.uint8)
      rc = self._L.mg_unit_generate(self._h, C.byref(d), _ptr(o1), _ptr(o2), nb.value, C.byref(nb), C.byref(nt), C.byref(nk))
    self._check(rc)
    return o1[:nb.value], o2[:nb.value], nt.value, nk.value, nb.value

  def wait_copies(self):
    self._check(self._L.mg_wait_copies(self._h))

  def unit_read(self, file, offset, nbytes, dst):
    """Enqueue the copy of bytes [offset, offset + nbytes) of file ``file`` of the most recent unit
    (generated with fetch=False) into ``dst`` (pinned uint8 array); valid after wait_copies()."""
    if dst.size < nbytes:
      raise ValueError('unit_read: destination too small')
    self._check(self._L.mg_unit_read_async(self._h, int(file), int(offset), int(nbytes), _ptr(dst)))
    return dst[:nbytes]

  def drain_async(self, sink, producer, unit):
    """Queue the most recent unit (generated with fetch=False) for streaming into ``sink`` as
    schedule unit ``unit``; returns at once, a thread of the context does the copies."""
    self._check(self._L.mg_unit_drain_async(self._h, sink._h, int(producer), int(unit)))

  def drain_wait(self):
    self._check(self._L.mg_drain_wait(self._h))

  # -- batches of small regions ------------------------------------------------------------------
  def build_batch(self, refs, bed_starts, seg_region, seg_variants):
    """refs: one uint8 array of reference bytes per region; bed_starts: their BED starts; seg_region[s] /
    seg_variants[s]: region index and VariantList of segment s (one chromosome copy of one region).
    -> BatchHandle with the segments' p_min / p_max (readgenerate.py:192)."""
    n_reg, n_seg = len(refs), len(seg_region)
    ref_off = np.zeros(n_reg + 1, dtype=np.int64)
    np.cumsum([len(r) for r in refs], out=ref_off[1:])
    ref = np.concatenate([np.asarray(r, dtype=np.uint8) for r in refs]) if n_reg else np.zeros(0, dtype=np.uint8)
    if ref.size == 0:
      ref = np.zeros(1, dtype=np.uint8)
    bed = np.ascontiguousarray(bed_starts, dtype=np.int64)
    sreg = np.ascontiguousarray(seg_region, dtype=np.int32)
    var_off = np.zeros(n_seg + 1, dtype=np.int64)
    np.cumsum([len(v) for v in seg_variants], out=var_off[1:])
    cat = lambda name, dt: np.ascontiguousarray(np.concatenate([getattr(v, name) for v in seg_variants]) if n_seg else np.zeros(0), dtype=dt)  # noqa: E731
    pos, op, oplen = cat('pos', np.int64), cat('op', np.uint8), cat('oplen', np.int64)
    alt_pool = np.concatenate([v.alt_pool[int(v.alt_off[0]):int(v.alt_off[len(v)])] for v in seg_variants if len(v)] +
                              [np.zeros(1, dtype=np.uint8)]).astype(np.uint8)
    alt_off = np.zeros(int(var_off[-1]) + 1, dtype=np.int64)
    base = 0
    for s, v in enumerate(seg_variants):                 # alt offsets into the concatenated pool
      if len(v):
        alt_off[var_off[s]:var_off[s + 1] + 1] = v.alt_off[:len(v) + 1] + (base - int(v.alt_off[0]))
        base += int(v.alt_off[len(v)] - v.alt_off[0])
    alt_off[-1] = base
    bid = C.c_int64(0)
    p_min, p_max = np.zeros(n_seg, dtype=np.int64), np.zeros(n_seg, dtype=np.int64)
    self._check(self._L.mg_batch_build(self._h, n_reg, _ptr(ref), _ptr(ref_off), _ptr(bed), n_seg, _ptr(sreg), _ptr(var_off), _ptr(pos),
                                       _ptr(op), _ptr(oplen), _ptr(alt_pool), _ptr(alt_off), C.byref(bid), _ptr(p_min), _ptr(p_max)))
    return BatchHandle(bid.value, p_min, p_max)

  def free_batch(self, batch):
    self._check(self._L.mg_batch_free(self._h, batch.id))

  def generate_batch(self, batch, unit_seg, unit_seed, unit_ncand, unit_index, sample, seg_chrom, seg_cpy, p, mode=MODE_PHILOX,
                     draws=None, corrupt=False, corrupt_seed=0, sink=None, producer=0):
    """All units of a batch in one launch sequence (mg_batch_generate).  seg_chrom / seg_cpy: chromosome
    name and copy index per SEGMENT; draws (deterministic mode): (ts, u_tlen, fo, cand_off) with the
    units' draws concatenated.  With ``sink`` the bytes are streamed into it as schedule units
    ``unit_index``; without, they stay on the device back to back (``unit_read``).
    -> (templates, bytes per file, per-unit bytes, per-unit templates)."""
    n = len(unit_seg)
    useg = np.ascontiguousarray(unit_seg, dtype=np.int32)
    useed = np.ascontiguousarray(np.asarray(unit_seed, dtype=np.int64) & 0xFFFFFFFF, dtype=np.uint32)
    ucand = np.ascontiguousarray(unit_ncand, dtype=np.int64)
    uidx = np.ascontiguousarray(unit_index, dtype=np.int64)
    names = [str(c).encode() for c in seg_chrom]
    chrom_off = np.zeros(len(names) + 1, dtype=np.int64)
    np.cumsum([len(c) for c in names], out=chrom_off[1:])
    chrom_pool = np.frombuffer(b''.join(names) + b'\0', dtype=np.uint8)
    scpy = np.ascontiguousarray(seg_cpy, dtype=np.int32)
    ts = u = fo = coff = None
    if mode == MODE_DET:
      ts, u, fo, coff = draws
      ts = np.ascontiguousarray(ts, dtype=np.int64); u = np.ascontiguousarray(u, dtype=np.float64)
      fo = np.ascontiguousarray(fo, dtype=np.int8); coff = np.ascontiguousarray(coff, dtype=np.int64)
    nt, nb = C.c_int64(0), C.c_int64(0)
    ub, ut = np.zeros(max(1, n), dtype=np.int64), np.zeros(max(1, n), dtype=np.int64)
    self._check(self._L.mg_batch_generate(self._h, batch.id, n, _ptr(useg), _ptr(useed), _ptr(ucand), _ptr(uidx), str(sample).encode(),
                                          _ptr(chrom_pool), _ptr(chrom_off), _ptr(scpy), float(p), int(mode), _ptr(ts), _ptr(u), _ptr(fo),
                                          _ptr(coff), int(bool(corrupt)), int(corrupt_seed) & 0xFFFFFFFF, sink._h if sink is not None else None,
                                          int(producer), C.byref(nt), C.byref(nb), _ptr(ub), _ptr(ut)))
    return nt.value, nb.value, ub[:n], ut[:n]

  # -- corruption --------------------------------------------------------------------------------
  def corrupt_fastq(self, fq1, fq2=None, mode=MODE_PHILOX, seed=0, draws=None, first_template=0, out=None, partial=False):
    """Whole-buffer corrupt-reads.  fq1/fq2: bytes or uint8 arrays of 4-line FASTQ records.
    draws (deterministic mode): (bq_rnd f64, call_rnd f64, base_rnd u8, draw_off i64[n_reads+1]).
    partial=True (chunked streaming): only the complete templates present in both buffers are
    processed and the consumed input byte counts are returned as a 4th / 5th value; first_template =
    templates processed by earlier chunks.  out: optional (pinned) output buffer pair."""
    a1, a2 = _u8(fq1), _u8(fq2)
    if not partial:
      if a1.size and a1[-1] != 10:
        a1 = np.concatenate([a1, np.array([10], dtype=np.uint8)])
      if a2 is not None and a2.size and a2[-1] != 10:
        a2 = np.concatenate([a2, np.array([10], dtype=np.uint8)])
    cap = int(a1.size + (a2.size if a2 is not None else 0)) + 64
    if out is not None:
      o1, o2 = out
      cap = min(o1.size, o2.size) if a2 is not None else o1.size
    else:
      o1 = np.empty(cap, dtype=np.uint8)
      o2 = np.empty(cap, dtype=np.uint8) if a2 is not None else None
    l1, l2, nt, c1, c2 = C.c_int64(0), C.c_int64(0), C.c_int64(0), C.c_int64(0), C.c_int64(0)
    bq = call = base = off = None
    if mode == MODE_DET:
      bq, call, base, off = draws
      bq = np.ascontiguousarray(bq, dtype=np.float64); call = np.ascontiguousarray(call, dtype=np.float64)
      base = np.ascontiguousarray(base, dtype=np.uint8); off = np.ascontiguousarray(off, dtype=np.int64)
    self._check(self._L.mg_corrupt_fastq(self._h, *_fastq_args(a1, a2), int(mode), int(seed) & 0xFFFFFFFF, _ptr(bq), _ptr(call), _ptr(base), _ptr(off),
                                         _ptr(o1), _ptr(o2) if a2 is not None else None, cap, C.byref(l1), C.byref(l2), C.byref(nt),
                                         int(first_template), C.byref(c1), C.byref(c2)))
    res = (o1[:l1.value], (o2[:l2.value] if a2 is not None else None), nt.value)
    return res + (c1.value, c2.value) if partial else res

  # -- profiling ---------------------------------------------------------------------------------
  def prof_reset(self):
    self._L.mg_prof_reset(self._h)

  def prof(self):
    ms, n, b, tl, pms = C.c_double(0), C.c_int64(0), C.c_int64(0), C.c_int64(0), C.c_double(0)
    self._L.mg_prof_get(self._h, C.byref(ms), C.byref(n), C.byref(b), C.byref(tl), C.byref(pms))
    return {'emit_ms': ms.value, 'emit_launches': n.value, 'emit_bytes': b.value, 'total_launches': tl.value, 'plan_ms': pms.value}


CHECK_CODES = {1: 'malformed qname', 2: 'chrom / copy / POS not among the loaded regions', 3: 'read length differs from rlen / CIGAR',
               4: "'=' segment differs from the reference", 5: "'X' base differs from the haplotype (or equals the reference)",
               6: 'inserted bases differ', 7: 'no insertion at that reference position', 8: 'unknown CIGAR op', 9: 'position out of range',
               10: "not a 4-line record with a bare '+' line"}


class Checker(object):
  """The god-aligner round trip on the device (mg_check_*): every read of a FASTQ pair of perfect
  reads is re-derived from its qname (chrom, copy, strand, POS, CIGAR), the reference and the node
  lists of the copies registered with ``add_copy``."""

  def __init__(self, engine):
    self.engine, self._L = engine, engine._L
    h = C.c_void_p()
    engine._check(self._L.mg_check_open(engine._h, C.byref(h)))
    self._h = h

  def add_copy(self, cp, chrom, cpy):
    self.engine._check(self._L.mg_check_add_copy(self._h, cp.id, str(chrom).encode(), int(cpy)))

  def check(self, fq1, fq2=None, max_report=64):
    """-> (templates checked, bad reads, [(file, record, code)], consumed bytes of fq1, of fq2)."""
    n, bad, c1, c2 = C.c_int64(0), C.c_int64(0), C.c_int64(0), C.c_int64(0)
    idx, code = np.zeros(max(1, max_report), dtype=np.int64), np.zeros(max(1, max_report), dtype=np.int32)
    self.engine._check(self._L.mg_check_fastq(self._h, *_fastq_args(fq1, fq2), C.byref(n), C.byref(bad), _ptr(idx), _ptr(code), int(max_report),
                                              C.byref(c1), C.byref(c2)))
    k = min(bad.value, max_report)
    rep = [(int(i // max(1, n.value)), int(i % max(1, n.value)), int(c)) for i, c in zip(idx[:k], code[:k])]
    return n.value, bad.value, rep, c1.value, c2.value

  def close(self):
    if self._h:
      self._L.mg_check_close(self._h)
      self._h = None


BAM_CODES = {1: "not a 4-line record with a bare '+' line", 2: 'malformed qname', 3: 'chrom is not a contig of the FASTA',
             4: 'read name longer than the 254 bytes BAM can hold', 5: 'read length differs from rlen / the CIGAR', 6: 'malformed CIGAR',
             7: 'alignment outside its contig'}


class BamWriter(object):
  """The god-aligner on the device (mg_bam_*): FASTQ chunks in, a coordinate-sorted BGZF BAM + BAI out.
  ``add`` encodes the complete templates of a chunk pair into the current sorted run; ``close`` sorts /
  merges and writes.  ``run_bytes``: device memory of one run (None: derived from free memory)."""

  def __init__(self, engine, bam, bai, contigs, header_text, sample, level=6, threads=1, run_bytes=None):
    self.engine, self._L = engine, engine._L
    names = [str(n).encode() for n, _ in contigs]
    self._names = (C.c_char_p * len(names))(*names)
    self._lens = np.ascontiguousarray([int(l) for _, l in contigs], dtype=np.int64)
    h = C.c_void_p()
    engine._check(self._L.mg_bam_open(engine._h, str(bam).encode(), str(bai).encode() if bai else None, len(names), self._names, _ptr(self._lens),
                                      header_text.encode(), str(sample).encode(), int(level), int(threads), int(run_bytes or 0), C.byref(h)))
    self._h = h

  def add(self, fq1, fq2=None):
    """-> (templates encoded, consumed bytes of fq1, of fq2).  A read the BAM cannot hold raises ValueError
    with (file, record in this chunk, reason) as ``args[1:]``."""
    n, c1, c2, bi, bc = C.c_int64(0), C.c_int64(0), C.c_int64(0), C.c_int64(-1), C.c_int32(0)
    rc = self._L.mg_bam_add(self._h, *_fastq_args(fq1, fq2), C.byref(n), C.byref(c1), C.byref(c2), C.byref(bi), C.byref(bc))
    if rc == _lib.MG_EVALUE and bi.value >= 0:
      nf = 2 if fq2 is not None else 1
      raise ValueError('not writable as a BAM record', bi.value % nf, bi.value // nf, BAM_CODES.get(bc.value, str(bc.value)))
    self.engine._check(rc)
    return n.value, c1.value, c2.value

  def close(self):
    """Sort / merge the last run, write BAM + BAI -> (records, sorted runs, {'device_ms', 'd2h_ms', 'write_ms'})."""
    n, runs, t = C.c_int64(0), C.c_int64(0), np.zeros(3, dtype=np.float64)
    h, self._h = self._h, None
    self.engine._check(self._L.mg_bam_close(h, C.byref(n), C.byref(runs), _ptr(t)))
    return n.value, runs.value, {'device_ms': t[0], 'd2h_ms': t[1], 'write_ms': t[2]}

  def abort(self):
    if self._h:
      self._L.mg_bam_abort(self._h)
      self._h = None


def write_sorted_bam(bam, bai, contigs, header_text, records, level=6, threads=1):
  """The BGZF writer + BAI builder without a device: ``records`` = encoded BAM records already in
  coordinate order (bytes).  -> number of records."""
  L = _lib.lib()
  names = (C.c_char_p * max(1, len(contigs)))(*[str(n).encode() for n, _ in contigs])
  lens = np.ascontiguousarray([int(l) for _, l in contigs] or [0], dtype=np.int64)
  buf = np.frombuffer(bytes(records) or b'\0', dtype=np.uint8)
  n = C.c_int64(0)
  rc = L.mg_bam_write_sorted(str(bam).encode(), str(bai).encode() if bai else None, len(contigs), names, _ptr(lens), header_text.encode(),
                             _ptr(buf), len(records), int(level), int(threads), C.byref(n))
  if rc != 0:
    raise (ValueError if rc == _lib.MG_EVALUE else RuntimeError)('mitty_b200: cannot write {} (rc={}): {}'.format(bam, rc, L.mg_last_error(None).decode()))
  return n.value


# mg_readmodel_bam / mg_alnerr_bam / mg_bam_scan errors (15-17: mg_alnerr_bam only): (what, whether bad_where is a record ordinal rather than a compressed offset)
BAM_READ_ERRORS = {1: ('not a gzip member', False), 2: ("a gzip member without a BGZF 'BC' extra subfield", False),
                   3: ('corrupt or truncated BGZF member', False), 4: ('CRC32 mismatch', False),
                   5: ('ISIZE differs from the inflated length', False), 6: ('not a BAM file (magic or header lengths)', False),
                   7: ('the file ends inside the BAM header', False), 8: ('block_size < 32', True),
                   9: ('the file ends inside the record', True), 10: ('read error', False),
                   11: ('read name overruns block_size', True), 12: ('CIGAR overruns block_size', True),
                   13: ('SEQ overruns block_size', True), 14: ('QUAL overruns block_size', True),
                   15: ("not a Mitty qname (fields, strand, pos, CIGAR or v_list)", True),
                   16: ('no read for this mate in the qname', True), 17: ('refID out of range', True)}
READ_MODEL_COUNTS = ('records', 'considered', 'counted', 'skip_flag', 'skip_mapq', 'skip_empty', 'skip_noqual', 'skip_long',
                     'inflated_bytes', 'compressed_bytes', 'eof_marker', 'chunks')
ALIGNMENT_COUNTS = ('records', 'analysed', 'skipped', 'unmapped', 'wrong_chrom', 'exact', 'clamped', 'strand_mismatch', 'no_variant_reads',
                    'variant_entries', 'inflated_bytes', 'compressed_bytes', 'eof_marker', 'chunks')


def bam_read_error(path, code, where):
  """The ValueError of a malformed BAM: names the record ordinal (0-based, file order) or the compressed offset."""
  what, is_record = BAM_READ_ERRORS.get(code, ('error {}'.format(code), False))
  return ValueError('{}: {} {}: {}'.format(path, 'record' if is_record else 'compressed offset', where, what))


def scan_bam(path, threads=1, chunk_bytes=64 << 20):
  """The BGZF BAM reader of ``read_model_counts`` without a device: inflate, check the framing and walk the
  record chain.  -> {'records', 'inflated_bytes', 'compressed_bytes', 'eof_marker'}; malformed input raises
  ValueError (record overruns inside block_size are checked on the device only)."""
  L = _lib.lib()
  st, bw, bc = np.zeros(4, dtype=np.int64), C.c_int64(-1), C.c_int32(0)
  rc = L.mg_bam_scan(str(path).encode(), int(threads), int(chunk_bytes), _ptr(st), C.byref(bw), C.byref(bc))
  if rc == _lib.MG_EVALUE and bc.value:
    raise bam_read_error(path, bc.value, bw.value)
  if rc != 0:
    raise (ValueError if rc == _lib.MG_EVALUE else RuntimeError)('mitty_b200: cannot read {} (rc={})'.format(path, rc))
  return dict(zip(('records', 'inflated_bytes', 'compressed_bytes', 'eof_marker'), (int(x) for x in st)))


class Sink(object):
  """The native output sink (mg_sink_*): writer threads inside the library put the units into the two
  FASTQ files in schedule order -- pwrite for regular files, ordered sequential writes for FIFOs /
  pipes, one gzip member per piece with ``gzip_level`` > 0.  ``slots`` page-locked slot pairs of
  ``chunk_bytes`` per producer (GPU) are the spill that lets GPUs run ahead of the files."""

  def __init__(self, path1, path2, n_units, n_producers=1, slots=4, chunk_bytes=64 << 20, gzip_level=0, threads=4, table=None, owner=True):
    """table: path of a shared unit table (a file on /dev/shm) when several PROCESSES write the same
    pair of regular files; ``owner`` creates it and truncates the outputs, the others open after a barrier."""
    self._L = _lib.lib()
    h = C.c_void_p()
    rc = self._L.mg_sink_create_shared(str(path1).encode(), str(path2).encode() if path2 is not None else None, int(n_units), int(n_producers),
                                       int(slots), int(chunk_bytes), int(gzip_level), int(threads),
                                       str(table).encode() if table is not None else None, int(bool(owner)), C.byref(h))
    if rc != 0:
      raise (OSError if rc == _lib.MG_EVALUE else RuntimeError)('mitty_b200: cannot create the output sink for {} / {} (rc={})'.format(path1, path2, rc))
    self._h = h
    self.chunk_bytes = int(chunk_bytes)

  def next_unit(self):
    """The next unit of the schedule that nobody has taken yet, or -1."""
    return int(self._L.mg_sink_next_unit(self._h))

  def unit_size(self, unit, nbytes):
    if self._L.mg_sink_unit_size(self._h, int(unit), int(nbytes)) != 0:
      raise RuntimeError('output sink: ' + self._L.mg_sink_error(self._h).decode())

  def put(self, producer, unit, offset, b1, b2=None):
    """Host bytes of one piece (test / corrupt-reads path): copied into a slot pair and committed."""
    p1, p2, slot = C.c_void_p(), C.c_void_p(), C.c_void_p()
    if self._L.mg_sink_acquire(self._h, int(producer), C.byref(p1), C.byref(p2), C.byref(slot)) != 0:
      raise RuntimeError('output sink: ' + self._L.mg_sink_error(self._h).decode())
    n = len(b1)
    C.memmove(p1.value, (C.c_char * n).from_buffer_copy(bytes(b1)) if not isinstance(b1, np.ndarray) else b1.ctypes.data, n)
    if b2 is not None and p2.value:
      C.memmove(p2.value, (C.c_char * n).from_buffer_copy(bytes(b2)) if not isinstance(b2, np.ndarray) else b2.ctypes.data, n)
    if self._L.mg_sink_commit(self._h, slot, int(unit), int(offset), n) != 0:
      raise RuntimeError('output sink: ' + self._L.mg_sink_error(self._h).decode())

  def put_stream(self, producer, units, sizes, b1, b2=None):
    """Host bytes of SEVERAL units back to back (what a batch of small units leaves the device as): their
    sizes are announced, then the stream travels in slot-sized pieces that run through unit boundaries
    (mg_sink_commit_multi).  units: ascending schedule indices; sizes: bytes per file of each."""
    units, sizes = np.asarray(units, dtype=np.int64), np.asarray(sizes, dtype=np.int64)
    base = np.zeros(units.size + 1, dtype=np.int64)
    np.cumsum(sizes, out=base[1:])
    for k, n in zip(units.tolist(), sizes.tolist()):
      self.unit_size(k, n)
    a1 = np.frombuffer(bytes(b1), dtype=np.uint8) if not isinstance(b1, np.ndarray) else b1
    a2 = None if b2 is None else (np.frombuffer(bytes(b2), dtype=np.uint8) if not isinstance(b2, np.ndarray) else b2)
    for lo in range(0, int(base[-1]), self.chunk_bytes):
      hi = min(lo + self.chunk_bytes, int(base[-1]))
      p1, p2, slot = C.c_void_p(), C.c_void_p(), C.c_void_p()
      if self._L.mg_sink_acquire(self._h, int(producer), C.byref(p1), C.byref(p2), C.byref(slot)) != 0:
        raise RuntimeError('output sink: ' + self._L.mg_sink_error(self._h).decode())
      C.memmove(p1.value, a1[lo:hi].ctypes.data, hi - lo)
      if a2 is not None and p2.value:
        C.memmove(p2.value, a2[lo:hi].ctypes.data, hi - lo)
      u0 = max(0, int(np.searchsorted(base, lo, side='right')) - 1)
      u1 = int(np.searchsorted(base, hi, side='left'))
      idx = np.arange(u0, min(u1, units.size))
      s0, s1 = np.maximum(base[idx], lo), np.minimum(base[idx + 1], hi)
      keep = s1 > s0
      idx, s0, s1 = idx[keep], s0[keep], s1[keep]
      un, uo, so, nb = (np.ascontiguousarray(x, dtype=np.int64) for x in (units[idx], s0 - base[idx], s0 - lo, s1 - s0))
      if self._L.mg_sink_commit_multi(self._h, slot, int(idx.size), _ptr(un), _ptr(uo), _ptr(so), _ptr(nb)) != 0:
        raise RuntimeError('output sink: ' + self._L.mg_sink_error(self._h).decode())

  def abort(self, why):
    if self._h:
      self._L.mg_sink_abort(self._h, str(why).encode()[:400])

  def close(self):
    """-> (bytes written to file 1, to file 2); raises if any write failed."""
    if not self._h:
      return None
    w1, w2 = C.c_int64(0), C.c_int64(0)
    err = self._L.mg_sink_error(self._h).decode()
    rc = self._L.mg_sink_close(self._h, C.byref(w1), C.byref(w2))
    self._h = None
    if rc != 0:
      raise IOError('mitty_b200: output sink failed: ' + (err or 'see stderr'))
    return w1.value, w2.value


def bind_host_thread_to_gpu(device):
  """Pin the calling host thread to the CPU cores next to ``device`` (NVML's affinity mask), so that
  the pinned FASTQ buffers it allocates afterwards land in that socket's memory and the device-to-host
  copies do not cross the inter-socket link.  Best effort: returns the core list or None."""
  import os
  try:
    import pynvml
    pynvml.nvmlInit()
    h = pynvml.nvmlDeviceGetHandleByIndex(int(device))
    n_words = (os.cpu_count() + 63) // 64
    mask = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
    cores = [64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1]
    allowed = os.sched_getaffinity(0)
    cores = [c for c in cores if c in allowed]
    if cores:
      os.sched_setaffinity(0, cores)
      return cores
  except Exception:
    pass
  return None


def device_count():
  return int(_lib.lib().mg_device_count())


_default = None


def default_engine():
  """Process-wide engine on cuda:0 for the plugin-style module functions."""
  global _default
  if _default is None:
    _default = Engine(0)
  return _default
