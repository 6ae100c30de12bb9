"""FASTQ input of corrupt-reads, check-reads and god-aligner: each file (plain, gzip, a FIFO or /dev/fd/N) is
read in chunks into one page-locked buffer, and the complete templates of a chunk are handed to the device while
the rest of each file is carried into the next chunk."""
import gzip
import io
from concurrent.futures import ThreadPoolExecutor

import numpy as np


def open_fastq(fname):
  """One open() per input: the inputs may be FIFOs or /dev/fd/N process substitutions
  (examples/reads/run.sh:13-16 of the reference feeds corrupt-reads from FIFOs), where a second
  open() blocks for ever or loses the bytes already read.  Nothing is read here: see sniff_gzip."""
  return io.open(fname, 'rb', buffering=1 << 20)      # BufferedReader: peek() does not consume


def sniff_gzip(fp):
  """gzip is recognised from the first bytes of the one open stream -- at the first READ, not at
  open time: a writer that opens its two FIFOs one after the other only starts to write once BOTH
  have a reader, so blocking on the first input's bytes before opening the second would deadlock."""
  if fp.peek(2)[:2] == b'\x1f\x8b':
    return gzip.GzipFile(fileobj=fp, mode='rb')
  return fp


class FastqStream(object):
  """A FASTQ file read in chunks into one (pinned) buffer; the unconsumed tail is carried over."""

  def __init__(self, fname, buf):
    self.fp = open_fastq(fname)
    self.sniffed = False
    self.buf, self.fill, self.eof = buf, 0, False

  def close(self):
    self.fp.close()

  def refill(self):
    if not self.sniffed:
      self.fp, self.sniffed = sniff_gzip(self.fp), True
    mv = memoryview(self.buf)
    while self.fill < self.buf.size and not self.eof:
      n = self.fp.readinto(mv[self.fill:])
      if not n:
        self.eof = True
        if self.fill and self.buf[self.fill - 1] != 10 and self.fill < self.buf.size:
          self.buf[self.fill] = 10; self.fill += 1           # last line without a newline
      else:
        self.fill += n

  def consume(self, n):
    rest = self.fill - n
    if rest:
      self.buf[:rest] = self.buf[n:self.fill].copy()
    self.fill = rest


def for_each_chunk(ins, step):
  """Runs ``step(a1, a2) -> (templates, consumed bytes of a1, of a2)`` over the chunks of one FastqStream or a
  pair (``a2`` is None for one) until a file is exhausted, then closes the streams.  The files are refilled in
  parallel: one writer that alternates between the two FIFOs of a pair would block on the one a serial reader is
  not reading."""
  try:
    with ThreadPoolExecutor(max_workers=len(ins)) as pool:
      while True:
        for fu in [pool.submit(st.refill) for st in ins]:
          fu.result()
        bufs = [st.buf[:st.fill] for st in ins]
        if any(b.size == 0 for b in bufs):
          return
        n, c1, c2 = step(bufs[0], bufs[1] if len(bufs) > 1 else None)
        if n == 0:
          if all(st.eof for st in ins):
            return
          raise ValueError('a FASTQ record is larger than the chunk size ({} bytes)'.format(ins[0].buf.size))
        for st, c in zip(ins, (c1, c2)):
          st.consume(c)
  finally:
    for st in ins:
      st.close()


def qname_of(buf, rec):
  """The name line ('@' included) of record ``rec`` of a FASTQ chunk (uint8 array)."""
  nl = np.flatnonzero(buf == 10)
  start = 0 if rec == 0 else int(nl[4 * rec - 1]) + 1
  end = int(nl[4 * rec]) if 4 * rec < nl.size else buf.size
  return bytes(buf[start:end]).decode(errors='replace')
