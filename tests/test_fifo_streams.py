"""The FASTQ input streams of corrupt-reads, check-reads and god-aligner must work on FIFOs and /dev/fd/N
process substitutions: the reference's own example feeds corrupt-reads from FIFOs (examples/reads/run.sh:13-16).
One open() per input, gzip sniffed from the first bytes of that same stream, both files of a pair read at once
(host logic; no GPU needed)."""
import gzip
import os
import threading

import numpy as np
import pytest

from mitty_b200.lib import fastqio
from mitty_b200.simulation import readcorrupt as rc
from tests import helpers as H

REC = b'@q%d\nACGTACGTAC\n+\n~~~~~~~~~~\n'


def _payload(n=5000):
  return b''.join(REC % k for k in range(n))


def _feed(path, data):
  with open(path, 'wb') as fp:          # blocks until the reader has opened the FIFO
    fp.write(data)


@pytest.mark.parametrize('gz', [False, True])
@pytest.mark.timeout(60)
def test_stream_reads_a_fifo_once(tmp_path, gz):
  data = _payload()
  fifo = str(tmp_path / 'in.fifo')
  os.mkfifo(fifo)
  t = threading.Thread(target=_feed, args=(fifo, gzip.compress(data) if gz else data), daemon=True)
  t.start()
  st = rc._Stream(fifo, np.zeros(4096, dtype=np.uint8))     # a second open() here would deadlock / lose bytes
  got = []
  while True:
    st.refill()
    if st.fill == 0:
      break
    got.append(st.buf[:st.fill].tobytes())
    st.consume(st.fill)
  st.close()
  t.join(timeout=10)
  assert b''.join(got) == data


@pytest.mark.timeout(60)
def test_stream_reads_dev_fd(tmp_path):
  """/dev/fd/N (what `<(cat < tf1)` expands to): re-opening a pipe's /dev/fd entry shares the read
  position with the first open, so sniffing with a separate open() would eat the first two bytes."""
  data = _payload(100)
  r, w = os.pipe()
  t = threading.Thread(target=lambda: (os.write(w, data), os.close(w)), daemon=True)
  t.start()
  st = rc._Stream('/dev/fd/{}'.format(r), np.zeros(1 << 16, dtype=np.uint8))
  st.refill()
  assert st.buf[:st.fill].tobytes() == data and st.eof
  st.close()
  os.close(r)
  t.join(timeout=10)


def _complete_templates(a1, a2):
  """A step that takes every template complete in both chunks: -> (n, consumed bytes of a1, of a2)."""
  n1, n2 = np.flatnonzero(a1 == 10), np.flatnonzero(a2 == 10)
  n = min(n1.size, n2.size) // 4
  return n, (int(n1[4 * n - 1]) + 1 if n else 0), (int(n2[4 * n - 1]) + 1 if n else 0)


@pytest.mark.timeout(60)
def test_chunk_loop_reads_a_fifo_pair_fed_by_one_writer(tmp_path):
  """A reader that refills one file until its buffer is full before it reads the other deadlocks on this feed."""
  data = [_payload(180000), b''.join(b'@t%d\nACGTACGTACGTACGT\n+\n~~~~~~~~~~~~~~~~\n' % k for k in range(180000))]
  assert all(len(d) > 5 << 20 for d in data)
  paths = [str(tmp_path / 'p1'), str(tmp_path / 'p2')]
  for p in paths:
    os.mkfifo(p)
  t = threading.Thread(target=H.feed_interleaved, args=(paths, data), daemon=True)
  t.start()
  ins = [fastqio.FastqStream(p, np.zeros(4 << 20, dtype=np.uint8)) for p in paths]
  got = [[], []]

  def step(a1, a2):
    n, c1, c2 = _complete_templates(a1, a2)
    got[0].append(a1[:c1].tobytes()); got[1].append(a2[:c2].tobytes())
    return n, c1, c2

  fastqio.for_each_chunk(ins, step)
  for st in ins:
    st.close()
  t.join(timeout=10)
  assert [b''.join(g) for g in got] == data
