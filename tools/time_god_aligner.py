"""god-aligner timing: a chr1-shaped 30x pair written by generate-reads --corrupt, then
  * the whole command (python entry point) at deflate levels 6 and 1,
  * its device phase (ingest + size + encode + sort + gather, host clock around synchronised work),
    the device-to-host copies (CUDA events) and the writing (BGZF deflate + BAI, host clock),
  * BGZF deflate alone (mg_bam_write_sorted over the decompressed records) at levels 1 and 6.
The card's name and power limit are printed with the numbers.

  python tools/time_god_aligner.py [--length 249250621] [--coverage 30] [--dir /dev/shm] [--threads N]
"""
import argparse
import os
import shutil
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))


def card():
  try:
    return subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True,
                          text=True, timeout=60).stdout.strip().splitlines()[0]
  except Exception as e:   # noqa: BLE001
    return 'unknown ({})'.format(e)


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--length', type=int, default=249250621)
  ap.add_argument('--coverage', type=float, default=30.0)
  ap.add_argument('--dir', default='/dev/shm')
  ap.add_argument('--threads', type=int, default=None)
  ap.add_argument('--deflate-mb', type=int, default=256, help='records deflated in the deflate-only measurement')
  a = ap.parse_args()
  import mitty_b200.benchmarking.god_aligner as ga
  import mitty_b200.simulation.illumina as il
  import mitty_b200.simulation.readgenerate as rg
  from mitty_b200 import synth
  from mitty_b200.engine import write_sorted_bam
  from mitty_b200.readmodels import load_model

  print('card:', card())
  threads = a.threads or ga.default_threads()
  d = tempfile.mkdtemp(prefix='god_aligner_', dir=a.dir)
  try:
    wl = synth.chr1_shaped(length=a.length)
    fa, vcf, bed = synth.write_workload(wl, os.path.join(d, 'w'))
    r1, r2 = os.path.join(d, 'r1.fq'), os.path.join(d, 'r2.fq')
    t = time.time()
    rg.process_multi_threaded(fa, vcf, wl['sample'], bed, il, load_model('hiseq-X-v2.5-Garvan.pkl'), a.coverage, r1, r2, threads=1, seed=7,
                              mode='philox', corrupt=True)
    fq_bytes = os.path.getsize(r1) + os.path.getsize(r2)
    print('workload: chr1-shaped {} bp, {}x, FASTQ pair {:.2f} GB written in {:.1f} s'.format(a.length, a.coverage, fq_bytes / 1e9, time.time() - t))
    bam = os.path.join(d, 'perfect.bam')
    for level in (6, 1):
      res = ga.process_multi_threaded(fa, bam, r1, r2, threads=threads, level=level)
      bam_bytes = os.path.getsize(bam)
      n = res['records']
      print('whole command, level {}, {} threads: {} records in {:.2f} s ({:.2f} M reads/s); BAM {:.2f} GB, {} run(s)'.format(
        level, threads, n, res['seconds'], n / res['seconds'] / 1e6, bam_bytes / 1e9, res['runs']))
      print('  device phase (H2D + index + size + encode + sort + gather): {:.1f} ms = {:.1f} M reads/s, {:.1f} GB/s of FASTQ in'.format(
        res['device_ms'], n / res['device_ms'] / 1e3, fq_bytes / res['device_ms'] / 1e6))
      print('  D2H of the sorted records: {:.1f} ms; writing (BGZF deflate + BAI): {:.1f} ms'.format(res['d2h_ms'], res['write_ms']))
    # deflate alone over the first --deflate-mb MB of the last BAM's records
    import gzip
    import struct
    with gzip.open(bam, 'rb') as g:
      raw = g.read((a.deflate_mb << 20) + (1 << 20))
    u = 8 + struct.unpack_from('<i', raw, 4)[0]
    n_ref = struct.unpack_from('<i', raw, u)[0]
    u += 4
    for _ in range(n_ref):
      u += 8 + struct.unpack_from('<i', raw, u)[0]
    r0 = u
    while u + 4 <= len(raw) and u + 4 + struct.unpack_from('<i', raw, u)[0] <= len(raw) and u - r0 < (a.deflate_mb << 20):
      u += 4 + struct.unpack_from('<i', raw, u)[0]
    recs = raw[r0:u]
    contigs = [(c, int(s.shape[0])) for c, s in wl['contigs']]
    for level in (1, 6):
      for th in sorted({1, threads}):
        t = time.time()
        write_sorted_bam(os.path.join(d, 'x.bam'), os.path.join(d, 'x.bam.bai'), contigs, ga.header_text(contigs, wl['sample']), recs, level=level, threads=th)
        dt = time.time() - t
        print('BGZF deflate alone, level {}, {} threads: {:.0f} MB/s of records ({:.2f} GB in {:.2f} s)'.format(level, th, len(recs) / dt / 1e6,
                                                                                                             len(recs) / 1e9, dt))
    print('card:', card())
  finally:
    shutil.rmtree(d, ignore_errors=True)


if __name__ == '__main__':
  main()
