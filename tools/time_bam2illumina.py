"""bam2illumina timing: a quarter-chr1 30x pair written by generate-reads --corrupt and aligned by god-aligner
--level 1 (as tools/time_god_aligner.py builds it), then `create-read-model bam2illumina` over that BAM:
  * the whole command (python entry point) with the box's cores and with fewer inflate threads,
  * its phases: reading the file, inflating (wall and per thread), host-to-device copies and the counting
    kernel (CUDA events), and the kernel's rate over the bytes it must read (fixed fields of every record
    plus the QUAL of the counted ones) and over the inflated stream.
The card's name and power limit are printed with the numbers.

  python tools/time_bam2illumina.py [--length 62312655] [--coverage 30] [--dir /dev/shm] [--threads N]
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
  ap.add_argument('--length', type=int, default=249250621 // 4)
  ap.add_argument('--coverage', type=float, default=30.0)
  ap.add_argument('--dir', default='/dev/shm')
  ap.add_argument('--threads', type=int, default=None)
  a = ap.parse_args()
  import numpy as np
  import mitty_b200.benchmarking.god_aligner as ga
  import mitty_b200.empirical.bam2illumina as b2i
  import mitty_b200.simulation.illumina as il
  import mitty_b200.simulation.readgenerate as rg
  from mitty_b200 import synth
  from mitty_b200.readmodels import load_model

  print('card:', card())
  threads = a.threads or b2i.default_threads()
  d = tempfile.mkdtemp(prefix='bam2illumina_', dir=a.dir)
  try:
    wl = synth.chr1_shaped(length=a.length)
    fa, vcf, bed = synth.write_workload(wl, os.path.join(d, 'w'))
    r1, r2 = os.path.join(d, 'r1.fq'), os.path.join(d, 'r2.fq')
    rg.process_multi_threaded(fa, vcf, wl['sample'], bed, il, load_model('hiseq-X-v2.5-Garvan.pkl'), a.coverage, r1, r2, threads=1, seed=7,
                              mode='philox', corrupt=True)
    bam = os.path.join(d, 'in.bam')
    res = ga.process_multi_threaded(fa, bam, r1, r2, threads=ga.default_threads(), level=1)
    os.unlink(r1)
    os.unlink(r2)
    print('workload: chr1-shaped {} bp, {}x, god-aligner level 1: {} records, BAM {:.2f} GB'.format(
      a.length, a.coverage, res['records'], os.path.getsize(bam) / 1e9))
    pkl = os.path.join(d, 'out.pkl')
    b2i.process_bam_parallel(bam, pkl, 'warm-up', threads=threads, every=1000)       # module load, page-locked buffers
    for th in sorted({threads, max(1, threads // 4), 1}, reverse=True):
      t = time.time()
      r = b2i.process_bam_parallel(bam, pkl, 'timed', threads=th)
      wall = time.time() - t
      tm = r['times']
      need = 36 * r['records'] + int(load_model(pkl)['r_cnt'])
      tms = np.asarray(r['thread_ms'])
      print('whole command, {} inflate threads: {:.2f} s for {} records ({:.2f} M records/s, {:.2f} GB/s inflated)'.format(
        th, wall, r['records'], r['records'] / wall / 1e6, r['inflated_bytes'] / wall / 1e9))
      print('  read {:.0f} ms; inflate (wall) {:.0f} ms = {:.2f} GB/s; per thread busy {:.0f}-{:.0f} ms (mean {:.0f}); record walk {:.0f} ms; '
            'H2D {:.0f} ms = {:.1f} GB/s; kernel {:.1f} ms over {} chunks; call total {:.0f} ms'.format(
              tm['read_ms'], tm['inflate_ms'], r['inflated_bytes'] / tm['inflate_ms'] / 1e6, tms.min(), tms.max(), tms.mean(), tm['walk_ms'], tm['h2d_ms'],
              r['inflated_bytes'] / max(tm['h2d_ms'], 1e-9) / 1e6, tm['kernel_ms'], r['chunks'], tm['total_ms']))
      print('  kernel: {:.1f} GB/s over the {:.2f} GB it must read (fixed fields + QUAL), {:.1f} GB/s over the {:.2f} GB inflated'.format(
        need / tm['kernel_ms'] / 1e6, need / 1e9, r['inflated_bytes'] / tm['kernel_ms'] / 1e6, r['inflated_bytes'] / 1e9))
    print('card:', card())
  finally:
    shutil.rmtree(d, ignore_errors=True)


if __name__ == '__main__':
  main()
