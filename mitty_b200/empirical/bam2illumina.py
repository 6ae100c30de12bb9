"""bam2illumina: an Illumina read model built from a BAM (``mitty/empirical/bam2illumina.py`` of the reference).

The counts -- qualities per (mate, cycle), read lengths, template lengths -- are made by
``Engine.read_model_counts``: host threads inflate the BGZF file, the device counts every record
(``k_readmodel``).  ``model_from_counts`` turns them into the model dict the reference pickles, and
``process_bam_parallel`` writes it as a ``.pkl`` that ``generate-reads`` and ``corrupt-reads`` load.

The rules (applied to every alignment record in file order, any sort order):
  - record k (0-based) is considered iff k % every == 0;
  - it is skipped when flag & 0xB04 (unmapped, secondary, QC-fail, supplementary), mapq < min_mq, l_seq == 0,
    QUAL is missing (0xFF) or l_seq > max_bp; duplicates are counted;
  - mate 1 iff (flag & 0xC1) == 0x81, else mate 0 (unpaired reads count as mate 0);
  - base i of SEQ is cycle l_seq - 1 - i on the reverse strand, else i (hard-clipped bases are not seen);
  - bq_mat[mate, cycle, min(qual, 93)] += 1; len_hist[l_seq] += 1;
  - tlen[|TLEN|] += 1 for a counted read with (flag & 0xC1) == 0x41 and |TLEN| < max_tlen (longer templates
    are dropped, not clipped).
"""
import logging
import os
import pickle
import tempfile
import time

import numpy as np

logger = logging.getLogger(__name__)


def default_threads():
  """Inflate threads: the box's cores, capped as the god-aligner caps its deflate threads."""
  return max(1, min(os.cpu_count() or 1, 64))


def model_from_counts(bq_mat, len_hist, tlen, description, min_mq=0):
  """The model dict of the reference's ``.pkl`` from the counts: ``cum_bq_mat`` = cumsum over qualities over
  the row total (0.0 on rows without counts), ``cum_tlen`` = cumsum(tlen) / tlen.sum(), ``r_cnt`` = bases
  counted, ``min_rlen`` / ``max_rlen`` = the shortest / longest read length present and ``mean_rlen`` the
  most frequent one, ties going to the longer (the reference's models carry the mode under this name)."""
  bq_mat = np.asarray(bq_mat, dtype=np.uint64)
  tlen = np.asarray(tlen, dtype=np.uint64)
  len_hist = np.asarray(len_hist, dtype=np.uint64)
  lens = np.nonzero(len_hist)[0]
  if lens.size == 0:
    raise ValueError('no read was counted')
  tot = bq_mat.sum(axis=2)
  with np.errstate(invalid='ignore', divide='ignore'):
    cum_bq = np.cumsum(bq_mat, axis=2) / tot[:, :, None]
    cum_tlen = np.cumsum(tlen) / tlen.sum()
  cum_bq[tot == 0] = 0.0
  if tlen.sum() == 0:
    cum_tlen[:] = 0.0
  mode = int(len_hist.size - 1 - np.argmax(len_hist[::-1]))
  return {'model_class': 'illumina', 'model_description': str(description), 'min_mq': int(min_mq),
          'bq_mat': bq_mat, 'cum_bq_mat': cum_bq, 'tlen': tlen, 'cum_tlen': cum_tlen,
          'r_cnt': int(bq_mat.sum()), 'min_rlen': int(lens[0]), 'max_rlen': int(lens[-1]), 'mean_rlen': mode}


def write_model(pkl, model):
  """Pickles ``model`` to a temporary file next to ``pkl`` and renames it into place, with the mode a plain
  ``open(pkl, 'wb')`` would give it (mkstemp creates the file 0600)."""
  d = os.path.dirname(os.path.abspath(pkl))
  fd, tmp = tempfile.mkstemp(prefix=os.path.basename(pkl) + '.', suffix='.tmp', dir=d)
  try:
    umask = os.umask(0)
    os.umask(umask)
    os.fchmod(fd, 0o666 & ~umask)
    with os.fdopen(fd, 'wb') as fp:
      pickle.dump(model, fp, protocol=pickle.HIGHEST_PROTOCOL)
    os.replace(tmp, pkl)
  except BaseException:
    os.unlink(tmp)
    raise


def process_bam_parallel(bam, pkl, description, every=1, min_mq=0, threads=None, max_bp=300, max_tlen=1000, device=0,
                         chunk_bytes=64 << 20):
  """Count ``bam`` (a BGZF BAM file or FIFO) and write the read model to ``pkl``.  ``threads``: host inflate
  threads (None: the box's cores); ``chunk_bytes``: inflated bytes per device chunk.  On malformed input (a
  ValueError naming the record ordinal or compressed offset), or when no read was counted, no ``pkl`` is
  written.  -> the counters of ``engine.READ_MODEL_COUNTS`` plus 'seconds', 'times' and 'thread_ms'."""
  from mitty_b200.engine import Engine
  t0 = time.time()
  threads = default_threads() if threads is None else max(1, int(threads))
  engine = Engine(device)
  try:
    res = engine.read_model_counts(bam, max_bp=max_bp, max_tlen=max_tlen, min_mq=min_mq, every=every, threads=threads, chunk_bytes=chunk_bytes)
  finally:
    engine.close()
  if not res['eof_marker']:
    logger.warning('%s has no BGZF EOF marker: the file may be truncated', bam)
  if res['counted'] == 0:
    raise ValueError('{}: no read was counted ({} records, {} considered)'.format(bam, res['records'], res['considered']))
  write_model(pkl, model_from_counts(res.pop('bq_mat'), res.pop('len_hist'), res.pop('tlen'), description, min_mq))
  res['seconds'] = time.time() - t0
  logger.debug('bam2illumina: {} of {} records counted in {:0.2f}s'.format(res['counted'], res['records'], res['seconds']))
  return res
