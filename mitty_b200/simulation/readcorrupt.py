"""corrupt-reads: ``mitty/simulation/readcorrupt.py`` on the GPU.

Same entry point as the reference (``multi_process``, readcorrupt.py:18).  The FASTQ pair is
indexed (newline scan), sized (exclusive scan) and corrupted on the device
(``k_nl_*``, ``k_corrupt_sizes``, ``k_corrupt_staged``; ``k_corrupt`` for the deterministic draws);
input qualities are discarded and read 1's name is written to both files, as the reference does
(readcorrupt.py:55, 113).

Page-locked memory: 2 input + 4 output buffers of ``chunk_bytes`` / 2 x ``chunk_bytes`` (2.5 GB with
the default 256 MB chunks; pass a smaller ``chunk_bytes`` on small hosts -- the result does not
depend on it).

Modes
  philox         production: Philox4x32-7 draws keyed by (seed, template index, file, cycle group);
                 one joint (quality, substitution) alias lookup per base (MgCorruptCtx, mg_core.cuh)
  deterministic  the single worker's numpy RandomState stream of the reference
                 (seed -> RandomState(seed).randint(SEED_MAX), readcorrupt.py:31,36,84) is drawn on
                 the host, read by read, and consumed on the device: byte-exact vs ``--threads 1``
"""
import logging
import time

import numpy as np

from mitty_b200.engine import MODE_DET, MODE_PHILOX, SEED_MAX, Engine
from mitty_b200.lib.fastqio import FastqStream, for_each_chunk

logger = logging.getLogger(__name__)

_Stream = FastqStream      # corrupt-reads' input stream under the name its FIFO / /dev/fd tests use


def seq_lengths(buf):
  """Lengths of the sequence lines of a 4-line-record FASTQ buffer (host side, numpy)."""
  nl = np.flatnonzero(buf == 10)
  n_rec = nl.size // 4
  return (nl[1:4 * n_rec:4] - nl[0:4 * n_rec:4] - 1).astype(np.int64)


def multi_process(read_module, read_model, fastq1_in, fastq1_out, fastq2_in=None, fastq2_out=None, processes=2, seed=7,
                  mode='philox', device=0, chunk_bytes=256 << 20):
  """Same signature as the reference (readcorrupt.py:18) plus keyword-only extras.  ``processes``
  is accepted for command-line compatibility (one GPU does all the work).  Note the reference
  passes the RAW model dict here (cli.py:155-157), and so does the CLI of this package.

  The files are read in chunks (``lib.fastqio``); the device corrupts the complete templates of each.
  The output does not depend on the chunk size.

  Page-locked host memory: one input buffer of ``chunk_bytes`` and two output buffers of twice that per file,
  i.e. 10 x chunk_bytes for a pair (2.5 GB at the default 256 MB; ``chunk_bytes`` scales it down)."""
  t0 = time.time()
  engine = Engine(device)
  cnt = 0
  try:
    rlen = read_model['mean_rlen'] if 'mean_rlen' in read_model else read_model['rlen']
    engine.load_model(read_model, rlen=rlen)
    paired = fastq2_in is not None
    ins = [FastqStream(f, engine.pinned(chunk_bytes)) for f in (fastq1_in, fastq2_in) if f is not None]
    # two output buffer sets: the files of chunk k are written (one thread per file) while chunk k+1
    # is read and corrupted
    outs = [(engine.pinned(2 * chunk_bytes + 64), engine.pinned(2 * chunk_bytes + 64) if paired else None) for _ in range(2)]
    pending = [[], []]
    from concurrent.futures import ThreadPoolExecutor
    pool = ThreadPoolExecutor(max_workers=4)
    k = 0
    rng = None
    if mode == 'deterministic':
      worker_seed = np.random.RandomState(seed).randint(SEED_MAX)   # worker 0, readcorrupt.py:31,36
      rng = np.random.RandomState(worker_seed)
    fps = [open(fastq1_out, 'wb')] + ([open(fastq2_out, 'wb')] if paired and fastq2_out is not None else [])

    def step(a1, a2):
      nonlocal k, cnt
      draws = None
      if rng is not None:
        l1 = seq_lengths(a1)
        if paired:
          l2 = seq_lengths(a2)
          n = min(l1.size, l2.size)
          lens = np.empty(2 * n, dtype=np.int64); lens[0::2] = l1[:n]; lens[1::2] = l2[:n]
        else:
          lens = l1
        draws = read_module.corrupt_draws(lens.tolist(), rng)
      for fu in pending[k]:                                   # this buffer set's previous writes
        fu.result()
      pending[k] = []
      o1, o2, n, c1, c2 = engine.corrupt_fastq(a1, a2, mode=MODE_DET if rng is not None else MODE_PHILOX, seed=seed, draws=draws,
                                               first_template=cnt, out=outs[k], partial=True)
      pending[k] = [pool.submit(fp.write, memoryview(o)) for fp, o in zip(fps, (o1, o2))]
      k ^= 1
      cnt += n
      return n, c1, c2

    try:
      for_each_chunk(ins, step)
    finally:
      for fu in pending[0] + pending[1]:
        fu.result()
      pool.shutdown(wait=True)
      for fp in fps:
        fp.close()
  finally:
    engine.close()
  t1 = time.time()
  logger.debug('Processed {} templates in {:0.2f}s ({:0.2f} t/s)'.format(cnt, t1 - t0, cnt / max(t1 - t0, 1e-9)))
