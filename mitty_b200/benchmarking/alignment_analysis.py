"""alignment-analysis: an aligner's BAM scored against the truth in Mitty's qnames (the reference's
``mitty/benchmarking/mq.py`` and ``derr.py``).

The counts are made by ``Engine.alignment_error_counts``: host threads inflate the BGZF file, the device
scores every record (``k_alnerr``).  ``write_csv`` writes the two matrices as ``PREFIX.mq.csv`` and
``PREFIX.vsize.csv``.  The rules (every record in file order, any sort order; DESIGN.md §11):
  - ``flag & 0x900`` (secondary, supplementary): skipped; QC-fail and duplicates are analysed;
  - the read is read 2 of the qname iff ``(flag & 0xC1) == 0x81``; its fields are those ``parse_qname`` gives it;
  - column ``unmapped`` for ``flag & 0x4`` or refID -1, ``wrong_chrom`` when the header name of refID is not the
    qname's chrom, else ``d = start(POS, CIGAR) - start(pos - 1, qname CIGAR)`` clamped to ``[-max_d, max_d]``,
    where ``start`` subtracts the leading run of S, H and I ops, so truth alignments and soft clips score 0;
  - ``mq[MAPQ, column] += 1``; ``vsize[clamp(v, -S-1, S+1) + S + 1, column] += 1`` per v_list entry, or the
    last row (``none``) for a read without variants.
"""
import logging
import os
import tempfile
import time

logger = logging.getLogger(__name__)


def csv_text(res, max_d, max_size):
  """-> (text of the mq file, text of the v_size file)."""
  cols = [str(d) for d in range(-max_d, max_d + 1)] + ['wrong_chrom', 'unmapped']

  def table(corner, labels, m):
    rows = [','.join([corner] + cols)]
    rows += [','.join([lab] + [str(int(x)) for x in row]) for lab, row in zip(labels, m.tolist())]
    return '\n'.join(rows) + '\n'

  v_labels = ['del>{}'.format(max_size)] + [str(v) for v in range(-max_size, max_size + 1)] + ['ins>{}'.format(max_size), 'none']
  return table('mq', [str(q) for q in range(256)], res['mq']), table('v_size', v_labels, res['vsize'])


def _write_atomic(path, text):
  """Writes ``text`` to a temporary file next to ``path`` and renames it into place, with the mode a plain
  ``open(path, 'w')`` would give it (mkstemp creates the file 0600)."""
  fd, tmp = tempfile.mkstemp(prefix=os.path.basename(path) + '.', suffix='.tmp', dir=os.path.dirname(os.path.abspath(path)))
  try:
    umask = os.umask(0)
    os.umask(umask)
    os.fchmod(fd, 0o666 & ~umask)
    with os.fdopen(fd, 'w') as fp:
      fp.write(text)
    return tmp
  except BaseException:
    os.unlink(tmp)
    raise


def write_csv(prefix, res):
  """Writes ``PREFIX.mq.csv`` and ``PREFIX.vsize.csv`` from the arrays of ``res`` (as ``process_bam`` returns
  them).  Both are written to temporary files next to the targets first and renamed only once both exist.
  -> the two paths."""
  max_d, max_size = (res['mq'].shape[1] - 3) // 2, (res['vsize'].shape[0] - 4) // 2
  paths = (prefix + '.mq.csv', prefix + '.vsize.csv')
  tmps = []
  try:
    for path, text in zip(paths, csv_text(res, max_d, max_size)):
      tmps.append(_write_atomic(path, text))
    for tmp, path in zip(tmps, paths):
      os.replace(tmp, path)
  except BaseException:
    for tmp in tmps:
      if os.path.exists(tmp):
        os.unlink(tmp)
    raise
  return paths


def read_csv(path):
  """-> (column labels, row labels, u64 matrix) of a CSV ``write_csv`` wrote."""
  import numpy as np
  lines = open(path).read().splitlines()
  cols = lines[0].split(',')[1:]
  rows = [ln.split(',') for ln in lines[1:]]
  return cols, [r[0] for r in rows], np.array([[int(x) for x in r[1:]] for r in rows], dtype=np.uint64).reshape(len(rows), len(cols))


def process_bam(bam, prefix=None, max_d=200, max_size=50, threads=None, device=0, chunk_bytes=64 << 20):
  """Score ``bam`` (a BGZF BAM file or FIFO) and, with ``prefix``, write the two CSVs.  ``threads``: host
  inflate threads (None: the box's cores); ``chunk_bytes``: inflated bytes per device chunk.  On malformed input
  (a ValueError naming the record ordinal or compressed offset) no CSV is written.  -> dict with 'mq', 'vsize',
  the counters of ``engine.ALIGNMENT_COUNTS``, 'seconds', 'times' and 'thread_ms'."""
  from mitty_b200.empirical.bam2illumina import default_threads
  from mitty_b200.engine import Engine
  t0 = time.time()
  threads = default_threads() if threads is None else max(1, int(threads))
  engine = Engine(device)
  try:
    res = engine.alignment_error_counts(bam, max_d=max_d, max_size=max_size, threads=threads, chunk_bytes=chunk_bytes)
  finally:
    engine.close()
  if not res['eof_marker']:
    logger.warning('%s has no BGZF EOF marker: the file may be truncated', bam)
  if prefix is not None:
    write_csv(prefix, res)
  res['seconds'] = time.time() - t0
  logger.debug('alignment-analysis: {} of {} records analysed in {:0.2f}s'.format(res['analysed'], res['records'], res['seconds']))
  return res
