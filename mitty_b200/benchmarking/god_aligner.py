"""god-aligner: the perfect alignments of a simulated FASTQ as a coordinate-sorted, indexed BAM
(``mitty/benchmarking/god_aligner.py`` of the reference, same entry point).

Every read becomes one BAM record at the POS / CIGAR its qname states (``parse_qname``): POS = qname pos
- 1, the qname's CIGAR ('>p:nI' becomes 'nI'), strand-1 reads reverse-complemented back and their
qualities reversed.  The FASTQ files are read in chunks through page-locked buffers (``lib.fastqio``); the device
parses, validates, encodes and sorts the records (``k_bam_size``, ``k_bam_encode``, ``k_radix_*``,
``k_gather_*``) in runs of at most ``run_bytes`` of device memory; host threads deflate the BGZF blocks
and build the BAI.  The bytes written do not depend on ``run_bytes``, the chunk size, ``threads`` or the
device."""
import logging
import os
import time

from mitty_b200.engine import BamWriter, Engine
from mitty_b200.lib.fastqio import FastqStream, for_each_chunk, qname_of
from mitty_b200.lib.vcfio import FastaFile

logger = logging.getLogger(__name__)

BAI_MAX_LEN = 1 << 29      # BAI bins address 2^29 bases


def default_threads():
  """Deflate threads: the box's cores, capped as the FASTQ sink caps its writer threads."""
  return max(1, min(os.cpu_count() or 1, 64))


def header_text(contigs, sample):
  return ('@HD\tVN:1.4\tSO:coordinate\n' + ''.join('@SQ\tSN:{}\tLN:{}\n'.format(n, l) for n, l in contigs) +
          '@RG\tID:{0}\tSM:{0}\tPL:ILLUMINA\n'.format(sample))


def sample_of(buf):
  """The sample field of the first qname of a FASTQ chunk ('@sample:worker:unit:serial|...')."""
  line = bytes(buf[:buf.size if buf.size < 4096 else 4096]).split(b'\n', 1)[0].decode(errors='replace')
  return line[1:].split('|', 1)[0].split(':', 1)[0].strip() if line.startswith('@') else ''


def process_multi_threaded(fasta, bam_fname, fastq1, fastq2=None, threads=None, device=0, level=6, run_bytes=None,
                           chunk_bytes=256 << 20, sample=None):
  """Write ``bam_fname`` and ``bam_fname + '.bai'`` from the FASTQ (pair).  ``threads``: host deflate threads;
  ``level``: BGZF deflate level (0 = stored blocks); ``run_bytes``: device memory of one sorted run (None:
  derived from free memory; smaller values only make more runs).  The sample of the ``@RG`` line is the
  first qname's.  A read the BAM cannot hold raises ValueError naming the record; then no BAM, no index
  and no temporary file is left.  -> {'records', 'runs', 'seconds', 'device_ms', 'd2h_ms', 'write_ms'}"""
  t0 = time.time()
  fa = FastaFile(fasta)
  contigs = [(n, fa.get_reference_length(n)) for n in fa.references]
  fa.close()
  bai = bam_fname + '.bai'
  if any(l > BAI_MAX_LEN for _, l in contigs):
    logger.warning('a contig is longer than 2^29 bases: BAI cannot index it, no %s is written', bai)
    bai = None
  if os.path.exists(bam_fname + '.bai') and bai is None:
    os.unlink(bam_fname + '.bai')
  threads = default_threads() if threads is None else max(1, int(threads))
  engine = Engine(device)
  bw = None
  try:
    ins = [FastqStream(f, engine.pinned(chunk_bytes)) for f in (fastq1, fastq2) if f is not None]
    templates = 0

    def writer(first):      # the BamWriter, opened at the first chunk: the @RG sample is its first qname's
      nonlocal bw
      if bw is None:
        s = sample_of(first) if sample is None else sample
        bw = BamWriter(engine, bam_fname, bai, contigs, header_text(contigs, s), s, level=level, threads=threads, run_bytes=run_bytes)
      return bw

    def step(a1, a2):
      nonlocal templates
      try:
        n, c1, c2 = writer(a1).add(a1, a2)
      except ValueError as e:
        if len(e.args) < 4:
          raise
        f, rec, why = e.args[1:]
        raise ValueError('{} record {}: {}: {}'.format(fastq1 if f == 0 else fastq2, templates + rec + 1, why, qname_of(a1 if f == 0 else a2, rec)))
      templates += n
      return n, c1, c2

    for_each_chunk(ins, step)
    records, runs, times = writer(ins[0].buf[:ins[0].fill]).close()      # an empty input still gets an empty BAM and BAI
    bw = None
  finally:
    if bw is not None:
      bw.abort()
    engine.close()
  res = {'records': records, 'runs': runs, 'seconds': time.time() - t0}
  res.update(times)
  logger.debug('god-aligner: {} records in {} sorted runs, {:0.2f}s'.format(records, runs, res['seconds']))
  return res
