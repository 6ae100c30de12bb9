"""check-reads: the god-aligner contract verified for every read (SURVEY.md 8f-1).

Mitty's ``god-aligner`` writes each read into a BAM at the POS / CIGAR its qname states
(mitty/benchmarking/god_aligner.py:141-183 over ``parse_qname``, readgenerate.py:259-291).  This
command proves that those qnames are true for a FASTQ pair of PERFECT reads: every read is re-derived
on the GPU from (chrom, copy, strand, POS, CIGAR) + FASTA + VCF + BED (``k_roundtrip_check``) and
compared with the bases in the file.  The files are read in chunks (``lib.fastqio``)."""
import logging
import time

import mitty_b200.lib.vcfio as vio
from mitty_b200.engine import CHECK_CODES, Checker, Engine
from mitty_b200.lib.fastqio import FastqStream, for_each_chunk, qname_of

logger = logging.getLogger(__name__)


def check_fastq(fasta_fname, vcf_fname, sample_name, bed_fname, fastq1, fastq2=None, device=0, chunk_bytes=256 << 20, max_report=20,
                drop_end_deletions=False):
  """-> {'templates', 'reads', 'bad', 'examples': [(file, record, reason, qname)], 'seconds'}"""
  from mitty_b200.simulation.readgenerate import _without_end_crossing_deletions
  t0 = time.time()
  vcf_df = vio.load_variant_file(vcf_fname, sample_name, bed_fname)
  fasta = vio.FastaFile(fasta_fname)
  engine = Engine(device)
  chk = None
  try:
    chk = Checker(engine)
    for r in vcf_df:
      region = r['region']
      rid = engine.load_region(fasta.fetch(reference=region[0], start=region[1], end=region[2]), region[1])
      for cpy, vl in enumerate(r['v']):
        vl, _ = _without_end_crossing_deletions(vl, region, drop_end_deletions)
        chk.add_copy(engine.build_copy(rid, vl), region[0], cpy)
    ins = [FastqStream(f, engine.pinned(chunk_bytes)) for f in (fastq1, fastq2) if f is not None]
    templates = bad = 0
    examples = []

    def step(a1, a2):
      nonlocal templates, bad
      n, nb, rep, c1, c2 = chk.check(a1, a2, max_report=max(0, max_report - len(examples)) or 1)
      for f, rec, code in rep:
        if len(examples) < max_report:
          examples.append((f + 1, templates + rec, CHECK_CODES.get(code, str(code)), qname_of(a1 if f == 0 else a2, rec)))
      templates += n; bad += nb
      return n, c1, c2

    for_each_chunk(ins, step)
    return {'templates': templates, 'reads': templates * len(ins), 'bad': bad, 'examples': examples, 'seconds': time.time() - t0}
  finally:
    if chk is not None:
      chk.close()
    engine.close()
