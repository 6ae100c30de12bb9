"""bench.py -- read pairs/s of the read-generation hot path (generate-reads + Illumina corruption).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload chr1|wgs] [--dump-outputs DIR]

Workload (config.workload)
  N = 1   BASELINE.json configs[2]: one chr1-shaped synthetic contig (249,250,621 bp, ~10 % N in long
          runs, ~330 k SNP/indel records, diploid), 30x, 2x150 (hiseq-X-v2.5-Garvan, the shipped 150-bp
          model; SURVEY.md 8d), production (Philox) mode with the corruption model fused into the emit
          kernel.  One STEP = the whole contig at 30x: both chromosome copies built, then all 4 work
          units (2 copies x 2 passes, ~22.6 M read pairs, ~17 GB of FASTQ).
  N > 1   BASELINE.json configs[3] (north_star's target run): the 3.1 Gb GRCh37-shaped genome, 24
          contigs, ~4 M variants, haploid X / Y, 30x: ~303 M pairs, ~228 GB of FASTQ per STEP, the work
          units SHARED by the ranks (strong scaling).  Units are independent: no collective on the
          data path; torch.distributed (NCCL) carries the barriers and the max / sum of the timings.

value   pairs/s with inputs resident in HBM (packed reference; variant arrays on the host side of
        mg_copy_build) and outputs left in HBM; CUDA events on the launch stream, max over ranks.
        With N > 1 the contigs are dealt to the ranks by LPT.
e2e     the same step through the PRODUCT's worker code (readgenerate.gpu_worker, what
        `generate-reads --threads N` runs per GPU) with HOST buffers: raw reference bytes H2D +
        packing, copy builds, units pulled in schedule order, every FASTQ byte D2H into page-locked
        slots and written IN SCHEDULE ORDER by the native output sink to the named target (one pair
        of files for all ranks: the ranks share the sink's unit table).  Wall clock between barriers.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODEL = 'hiseq-X-v2.5-Garvan.pkl'
COVERAGE = 30.0
SLICE = 10000000       # C-port CPU sample: one 10 Mb slice of the same contig
REF_SLICE = 250000     # real-reference CPU sample: a 250 kb slice (the reference is pure Python)
REF_DIR = os.path.join(ROOT, 'baseline', '_ref')


def parse():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=5)
  ap.add_argument('--warmup', type=int, default=3)
  ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
  ap.add_argument('--contig-len', type=int, default=249250621)
  ap.add_argument('--seed', type=int, default=7)
  ap.add_argument('--no-e2e', action='store_true')
  ap.add_argument('--no-cpu-baseline', action='store_true')
  ap.add_argument('--perfect', action='store_true', help='perfect reads only (no fused corruption)')
  ap.add_argument('--workload', default=None, choices=['chr1', 'wgs'], help="default: chr1 (configs[2]) on one GPU, wgs (configs[3], strong scaling) on several")
  ap.add_argument('--scale', type=float, default=1.0, help='length scale of the wgs workload')
  ap.add_argument('--sink', default=None, help="e2e target directory, or /dev/null (default: /dev/shm when a step's FASTQ fits, else /dev/null)")
  ap.add_argument('--e2e-steps', type=int, default=None, help='timed e2e steps (default: --steps, capped so that the leg stays within minutes)')
  ap.add_argument('--mode', default='generate-reads', choices=['generate-reads', 'corrupt-reads'], help="'corrupt-reads': the standalone corrupt kernel over a resident FASTQ pair (second-figure roofline, 1480 B/pair)")
  ap.add_argument('--soft-masked', action='store_true', help='chr1 workload with half of the bases in lower-case stretches (not the headline configuration)')
  ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                  help='after the timed steps, write what the last one computed as DIR/<name>.npy (see OutputSample); with several ranks, DIR/rank<r>/')
  a = ap.parse_args()
  if a.steps < 1 or a.warmup < 0:
    ap.error('--steps must be at least 1 and --warmup at least 0')
  if a.dump_outputs and a.impl != 'b200':
    ap.error('--dump-outputs records the outputs of this project (--impl b200)')
  world = int(os.environ.get('WORLD_SIZE', '1'))
  if a.workload is None:
    a.workload = 'wgs' if max(world, a.gpus) > 1 else 'chr1'
  return a


class ClockSampler(object):
  """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
  Q = 'index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

  def __init__(self, index):
    self.index, self.rows, self.p = index, [], None

  def start(self):
    try:
      self.p = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits', '-lms', '25'],
                                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      self.t = threading.Thread(target=self._read, daemon=True); self.t.start()
    except Exception:
      self.p = None

  def _read(self):
    for line in self.p.stdout:
      self.rows.append((time.perf_counter(), [x.strip() for x in line.split(',')]))

  def mark(self):
    """start of the timed region (the sampler itself is started before the warm-up: nvidia-smi takes
    longer to start than a short timed region lasts)"""
    self.t_mark = time.perf_counter()

  def stop(self):
    if self.p is None:
      return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
    self.p.terminate()
    try:
      self.p.wait(timeout=5)
    except Exception:
      self.p.kill()
    sm, mx, reasons = [], [], set()
    rows = [r for t, r in self.rows if t >= getattr(self, 't_mark', 0.0)]
    window = 'timed region'
    if not rows:   # no sample fell into a very short timed region: use the warm-up samples (same load)
      rows, window = [r for t, r in self.rows], 'warm-up + timed region'
    for r in rows:
      try:
        sm.append(float(r[1])); mx.append(float(r[2]))
        for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[4:8]):
          if v.lower().startswith('active'):
            reasons.add(name)
      except Exception:
        pass
    return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
            'reasons': sorted(reasons), 'samples': len(sm), 'window': window}


def measured_peak():
  p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(p):
    try:
      return float(json.load(open(p))['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs, copy bandwidth)'
    except Exception:
      pass
  return 6650.0, 'fallback (B200_PROFILING.md)'


def make_chr1(args, seed_off=0):
  from mitty_b200 import synth
  length = args.contig_len
  scale = length / 249250621.0
  wl = synth.chr1_shaped(seed=args.seed + seed_off, length=length, n_runs=max(3, int(39 * scale)))
  if getattr(args, 'soft_masked', False):        # repeat-masker style: alternating stretches, mean length 300
    seq = wl['contigs'][0][1]
    edges = np.cumsum(np.random.RandomState(5).geometric(1.0 / 300.0, size=2 * length // 300 + 64))
    edges = edges[edges < length]
    low = (np.searchsorted(edges, np.arange(length), side='right') & 1).astype(bool) & (seq != ord('N'))
    seq[low] |= 0x20
  return wl


# ---- CPU baselines -----------------------------------------------------------------------------------

def _cpu_unit(job):
  """One oracle work unit on a slice: generate-reads + corrupt-reads (single thread, C port)."""
  import oracle
  ref, start, vl_arrays, rm_small, seed, cum_bq = job
  cv = oracle.CopyVariants(*vl_arrays)
  p_min, p_max, _ = oracle.node_span(ref, start + 1, cv)
  t0 = time.perf_counter()
  ts, te, fo = oracle.templates(rm_small['p'], rm_small['rlen'], rm_small['cum_tlen'], p_min, p_max, seed)
  f1, f2, n = oracle.generate_unit(ref, start + 1, cv, rm_small['rlen'], ts, te, fo, 'S:0:0', '1', 0)
  c1, c2, _ = oracle.corrupt_fastq(cum_bq, seed, f1, f2)
  return n, time.perf_counter() - t0


def _slice_variants(table, region, cpy):
  from mitty_b200.lib import vcfio
  start, end = region[1], region[2]
  vl = vcfio.from_variant_table(table, region)['v'][cpy]
  keep = (vl.pos > start + 1000) & (vl.pos < end - 1000)       # no deletion across the slice ends
  return vl, np.flatnonzero(keep)


def cpu_jobs(wl, n_jobs):
  import mitty_b200.simulation.illumina as il
  from mitty_b200.readmodels import load_model
  model = load_model(MODEL)
  rm = il.read_model_params(model, COVERAGE)
  rm_small = {'p': rm['p'], 'rlen': int(rm['rlen']), 'cum_tlen': np.asarray(rm['cum_tlen'])}
  seq = wl['contigs'][0][1]
  length = seq.shape[0]
  sl = min(SLICE, length)
  jobs = []
  for k in range(n_jobs):
    # slices are taken from the non-N part of the contig, round robin
    start = int((length // 3 + k * sl) % max(1, length - sl))
    vl, idx = _slice_variants(wl['tables'][0], (wl['contigs'][0][0], start, start + sl), k % 2)
    alts = [vl.alt_pool[vl.alt_off[i]:vl.alt_off[i + 1]].tobytes().decode() for i in idx]
    jobs.append((np.ascontiguousarray(seq[start:start + sl]), start, (vl.pos[idx], vl.op[idx], vl.oplen[idx], alts), rm_small,
                 1000 + k, np.asarray(model['cum_bq_mat'])))
  return jobs, sl


def port_baseline(wl, procs):
  """The C restatement of the reference algorithm (oracle/), `procs` processes x one slice each."""
  import multiprocessing as mp
  import oracle
  oracle.build()
  jobs, sl = cpu_jobs(wl, procs)
  t0 = time.perf_counter()
  if procs == 1:
    res = [_cpu_unit(jobs[0])]
  else:
    with mp.get_context('fork').Pool(procs) as pool:
      res = pool.map(_cpu_unit, jobs)
  wall = time.perf_counter() - t0
  return sum(r[0] for r in res), wall, sl


class ReferenceRunner(object):
  """The UNMODIFIED reference (baseline/_ref: `pip install --target` of /root/reference + the pysam
  I/O stand-in, oracle/install_reference.py) on a slice of the workload: its own
  generate-reads followed by its own corrupt-reads, `--threads T` each, files on local disk."""

  def __init__(self, wl, threads):
    import tempfile
    from mitty_b200 import synth
    self.threads = threads
    seq = wl['contigs'][0][1]
    name = wl['contigs'][0][0]
    length = seq.shape[0]
    sl = min(REF_SLICE, length)
    start = int(length // 3)
    table = wl['tables'][0]
    keep = (table.pos > start + 1000) & (table.pos + 50 < start + sl - 1000)
    sub = synth._subset(table, keep)
    sub = synth.VariantTable(sub.chrom, sub.pos - start, sub.ref_pool, sub.ref_off, sub.alt_pool, sub.alt_off, sub.gt)
    small = {'contigs': [(name, np.ascontiguousarray(seq[start:start + sl]))], 'tables': [sub], 'regions': [(name, 0, sl)], 'sample': wl['sample']}
    self.dir = tempfile.mkdtemp(prefix='mitty_ref_bench_')
    self.fa, self.vcf, self.bed = synth.write_workload(small, os.path.join(self.dir, 'slice'))
    self.sample, self.slice = wl['sample'], sl
    sys.path.insert(0, REF_DIR)
    import warnings
    warnings.filterwarnings('ignore')
    import pickle
    import mitty.simulation.illumina as ril
    import mitty.simulation.readcorrupt as rrc
    import mitty.simulation.readgenerate as rrg
    self.il, self.rc, self.rg = ril, rrc, rrg
    self.model = pickle.load(open(os.path.join(REF_DIR, 'mitty', 'data', 'readmodels', MODEL), 'rb'))

  def step(self, seed):
    p = {k: os.path.join(self.dir, k + '.fq') for k in ('r1', 'r2', 'c1', 'c2')}
    t0 = time.perf_counter()
    self.rg.process_multi_threaded(self.fa, self.vcf, self.sample, self.bed, self.il, self.model, COVERAGE, p['r1'], p['r2'],
                                   threads=self.threads, seed=seed)
    t1 = time.perf_counter()
    self.rc.multi_process(self.il, self.model, p['r1'], p['c1'], p['r2'], p['c2'], processes=self.threads, seed=seed)
    t2 = time.perf_counter()
    with open(p['c1'], 'rb') as fp:
      pairs = fp.read().count(b'\n') // 4
    return pairs, t2 - t0, t1 - t0, t2 - t1

  def close(self):
    import shutil
    shutil.rmtree(self.dir, ignore_errors=True)


def reference_available():
  return os.path.isdir(os.path.join(REF_DIR, 'mitty')) and os.path.exists(os.path.join(REF_DIR, 'pysam.py'))


def run_reference(args):
  """--impl reference: the reference's own CPU implementation of the path on the box's host cores."""
  rank = int(os.environ.get('RANK', '0'))
  if rank != 0:
    return
  cores = os.cpu_count() or 1
  wl = make_chr1(args)
  line = {'impl': 'reference', 'metric': 'read pairs/sec (2x150, FASTQ-formatted, corrupted)', 'unit': 'pairs/s', 'n_gpus': args.gpus,
          'steps': args.steps, 'warmup': args.warmup, 'higher_is_better': True, 'scaling': 'strong' if args.workload == 'wgs' else 'weak',
          'vs_baseline': None, 'dtype': 'u8', 'data': 'synthetic', 'config': config_dict(args), 'gpu_launches': 0}
  # the C port on all cores, as a second figure (it is ~100x faster than the Python reference)
  procs = max(1, min(cores, 64))
  pn, pwall, psl = port_baseline(wl, procs)
  port = {'value': pn / pwall, 'unit': 'pairs/s', 'cores': procs, 'kind': 'port',
          'sample': '{} processes x one {} Mb-slice work unit (generate + corrupt), C restatement of the reference (oracle/)'.format(procs, psl // 1000000)}
  if reference_available():
    T = max(1, min(cores, 32))
    rr = ReferenceRunner(wl, T)
    times, pairs, gen_s, cor_s = [], 0, 0.0, 0.0
    for s in range(args.warmup + args.steps):
      n, wall, tg, tc = rr.step(args.seed + s)
      if s >= args.warmup:
        times.append(wall); pairs += n; gen_s += tg; cor_s += tc
    rr.close()
    value = pairs / sum(times)
    sample = ('mitty generate-reads --threads {T} then mitty corrupt-reads --threads {T} (unmodified reference, baseline/_ref) on a {kb} kb slice '
              'of the contig, ~{p} pairs per step; generate {g:.0f} / corrupt {c:.0f} pairs/s').format(
                T=T, kb=rr.slice // 1000, p=pairs // max(1, args.steps), g=pairs / max(gen_s, 1e-9), c=pairs / max(cor_s, 1e-9))
    line.update(value=value, ms_per_step=1e3 * sum(times) / len(times),
                cpu_baseline={'value': value, 'unit': 'pairs/s', 'cores': T, 'nproc': cores, 'kind': 'reference', 'sample': sample, 'port': port})
  else:
    line.update(value=port['value'], ms_per_step=1e3 * pwall, cpu_baseline=dict(port, note='baseline/_ref missing: C port only'))
  line['e2e'] = {'value': line['value'], 'unit': 'pairs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
  emit(line)


def config_dict(args):
  if args.workload == 'wgs':
    return {'workload': 'configs[3]: GRCh37-shaped synthetic genome (24 contigs, lengths x {}, ~8% N, ~4 M variants, diploid autosomes, haploid X/Y), '
                        '30x paired 2x150, Philox mode{}, work units shared by the ranks (strong scaling)'.format(args.scale, '' if args.perfect else ' + fused Illumina corruption'),
            'read_model': MODEL + ' (mean_rlen 150)', 'coverage': COVERAGE, 'seed': args.seed,
            'parallelism': 'units independent, no collective; value: contigs dealt by LPT; e2e: units pulled in schedule order from the shared sink',
            'l2': 'every unit streams its FASTQ through L2 (>> 126 MB for the large contigs)'}
  return {'workload': 'configs[2]: chr1-shaped synthetic contig ({} bp, ~10% N, GIAB-density diploid VCF), 30x paired 2x150, '
                      'Philox mode{}{}'.format(args.contig_len, '' if args.perfect else ' + fused Illumina corruption',
                                               ', SOFT-MASKED variant (half of the bases lower case)' if getattr(args, 'soft_masked', False) else ''),
          'read_model': MODEL + ' (mean_rlen 150)', 'coverage': COVERAGE, 'units_per_step': 4, 'seed': args.seed,
          'parallelism': 'one contig per GPU, units independent, no collective',
          'l2': 'each unit streams ~4.2 GB of FASTQ through L2 (>> 126 MB), so nothing is re-read warm between timed units'}


# ---- the engine --------------------------------------------------------------------------------------

_REAL_STDOUT = None


def _guard_stdout():
  """The contract is ONE JSON line on stdout: anything a library prints there (NCCL's version
  banner, for one) is sent to stderr instead; emit() writes to the real stdout."""
  global _REAL_STDOUT
  if _REAL_STDOUT is None:
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def emit(line):
  data = (json.dumps(line) + '\n').encode()
  if _REAL_STDOUT is None:
    sys.stdout.write(data.decode()); sys.stdout.flush()
  else:
    os.write(_REAL_STDOUT, data)


def pick_sink(args, bytes_per_step):
  """-> (path1, path2, description).  /dev/shm when one step's FASTQ fits with room to spare (the
  files are rewritten every step), else /dev/null (the writer threads still receive every byte)."""
  want = args.sink
  if want is None:
    try:
      st = os.statvfs('/dev/shm')
      free = st.f_bavail * st.f_frsize
      avail = free
      for ln in open('/proc/meminfo'):
        if ln.startswith('MemAvailable:'):
          avail = int(ln.split()[1]) * 1024
      want = '/dev/shm' if min(free, avail) > 1.25 * bytes_per_step + (24 << 30) else '/dev/null'
    except OSError:
      want = '/dev/null'
  if want == '/dev/null':
    return '/dev/null', '/dev/null', '/dev/null (page-locked slots -> native writer threads, bytes discarded by the kernel)'
  tag = os.environ.get('MASTER_PORT', str(os.getppid()))
  return (os.path.join(want, 'mitty_b200_bench_{}.1.fq'.format(tag)), os.path.join(want, 'mitty_b200_bench_{}.2.fq'.format(tag)),
          '{} (tmpfs files; the native writer threads copy every piece to its final offset through a shared mapping)'.format(want))


DUMP_BYTES = 12 << 20    # FASTQ bytes sampled from one step for --dump-outputs, shared by the ranks: 48 MB as float32
DUMP_WINDOWS = 8         # sampled windows per unit and FASTQ file
DUMP_SEED = 20240        # fixes where in a unit the windows lie


class OutputSample(object):
  """--dump-outputs: what the timed path hands its caller in its last step, as .npy files on which two
  builds can be compared.  A step writes GBs of FASTQ, so of each FASTQ file of each unit (a work unit
  of generate-reads, an input chunk of corrupt-reads) DUMP_WINDOWS windows are copied, at fixed seeded
  fractions of the file's length: equal outputs are sampled at equal offsets.  With several ranks each
  rank writes its own units under DIR/rank<r>/ and the ranks split DUMP_BYTES.

    unit<k>_fastq<m>.npy   float32 [DUMP_WINDOWS, width]  the byte values of the windows of file m (1, 2)
    window_offsets.npy     float64 [units, 2, DUMP_WINDOWS]  where the windows start
    unit_bytes.npy         float64 [units, 2]  bytes of each file
    unit_<count>.npy       float64 [units]  the counts the path returns per unit (templates, ...)
  """

  def __init__(self, path, max_units, alloc):
    world = int(os.environ.get('WORLD_SIZE', '1'))
    self.path = path if world == 1 else os.path.join(path, 'rank{}'.format(int(os.environ.get('RANK', '0'))))
    self.max_units = max_units
    self.width = max(1, DUMP_BYTES // world // (2 * DUMP_WINDOWS * max(1, max_units)))
    self.buf = alloc(2 * DUMP_WINDOWS * self.width * max(1, max_units))
    self.frac = np.sort(np.random.RandomState(DUMP_SEED).random_sample(DUMP_WINDOWS))
    self.units = []

  def take(self, read, sizes, **counts):
    """One unit: read(m, offset, nbytes, dst) copies bytes of its file m (0, 1), of sizes[m] bytes, into dst."""
    k = len(self.units)
    if k == self.max_units:
      raise RuntimeError('--dump-outputs: more than the {} units planned for'.format(self.max_units))
    windows = []
    for m in (0, 1):
      w = min(self.width, int(sizes[m]))
      offs = (self.frac * (int(sizes[m]) - w)).astype(np.int64)
      for j, o in enumerate(offs):
        start = ((2 * k + m) * DUMP_WINDOWS + j) * self.width
        read(m, int(o), w, self.buf[start:start + w])
      windows.append((offs, w))
    self.units.append((counts, sizes, windows))

  def write(self):
    os.makedirs(self.path, exist_ok=True)
    for k, (_, _, windows) in enumerate(self.units):
      for m, (_, w) in enumerate(windows):
        start = (2 * k + m) * DUMP_WINDOWS * self.width
        rows = self.buf[start:start + DUMP_WINDOWS * self.width].reshape(DUMP_WINDOWS, self.width)[:, :w]
        np.save(os.path.join(self.path, 'unit{}_fastq{}.npy'.format(k, m + 1)), rows.astype(np.float32))
    np.save(os.path.join(self.path, 'window_offsets.npy'), np.array([[offs for offs, _ in u[2]] for u in self.units], dtype=np.float64))
    np.save(os.path.join(self.path, 'unit_bytes.npy'), np.array([u[1] for u in self.units], dtype=np.float64))
    for name in (self.units[0][0] if self.units else {}):
      np.save(os.path.join(self.path, 'unit_{}.npy'.format(name)), np.array([u[0][name] for u in self.units], dtype=np.float64))


def main():
  if os.environ.get('MG_BENCH_LOG'):
    import logging
    logging.basicConfig(level=getattr(logging, os.environ['MG_BENCH_LOG'].upper(), logging.INFO))
  args = parse()
  _guard_stdout()
  if args.impl == 'reference':
    return run_reference(args)

  import torch
  import torch.distributed as dist
  rank = int(os.environ.get('RANK', '0'))
  local = int(os.environ.get('LOCAL_RANK', '0'))
  world = int(os.environ.get('WORLD_SIZE', '1'))
  torch.cuda.set_device(local)
  from mitty_b200.engine import bind_host_thread_to_gpu
  numa_cores = bind_host_thread_to_gpu(local) if world > 1 else None   # pinned buffers next to the GPU
  if world > 1:
    dist.init_process_group('nccl', device_id=torch.device('cuda', local))

  import mitty_b200.simulation.illumina as il
  import mitty_b200.simulation.readgenerate as rg
  from mitty_b200 import multigpu, synth
  from mitty_b200.engine import Engine, Sink
  from mitty_b200.lib import vcfio
  from mitty_b200.readmodels import load_model

  model = load_model(MODEL)
  rm = il.read_model_params(model, COVERAGE)
  L = int(rm['rlen'])
  stream = torch.cuda.Stream()
  eng = Engine(local, stream=stream.cuda_stream)
  eng.load_model(rm)
  corrupt = not args.perfect

  if args.mode == 'corrupt-reads':
    return bench_corrupt_reads(args, eng, rm, model)

  # ---- the workload: every rank holds all of it (the e2e leg hands units out dynamically)
  if args.workload == 'wgs':
    wl = synth.grch37_shaped(scale=args.scale, seed=args.seed)
  else:
    wl = make_chr1(args, 101 * rank if world > 1 else 0)
  tables = {t.chrom: t for t in wl['tables']}
  contigs = dict(wl['contigs'])
  vcf_df = [vcfio.from_variant_table(tables[region[0]], region) for region in wl['regions']]
  refs = {region: np.ascontiguousarray(contigs[region[0]][region[1]:region[2]]) for region in wl['regions']}
  # the step's host inputs (the reference bytes of every region) live in page-locked host memory, as the timing contract
  # asks: the H2D copy inside the timed region then runs at the link's speed instead of through the driver's staging buffer
  pinned_keep = []
  if sum(a.nbytes for a in refs.values()) <= (4 << 30):
    for region, a in list(refs.items()):
      t = torch.empty(max(1, a.size), dtype=torch.uint8).pin_memory()
      v = t.numpy()[:a.size]
      v[:] = a
      refs[region] = v
      pinned_keep.append(t)
  fetch_ref = lambda region: refs[region]  # noqa: E731
  if args.workload == 'wgs':
    mine = multigpu.assign_units([r[2] - r[1] for r in wl['regions']], world)[rank]       # value leg: contigs by LPT
  else:
    mine = [0]

  def value_step(seed, rids, sample=None):
    """The rank's contigs: copies built from the resident packed region, then copies x passes units,
    outputs left in HBM (with `sample`, windows of them are also copied to the host).  -> (pairs, fastq bytes)"""
    pairs = nbytes = 0
    k = 0
    for ci, rid in zip(mine, rids):
      region_, r_ = wl['regions'][ci], vcf_df[ci]
      copies = [eng.build_copy(rid, vl) for vl in r_['v']]
      for cpy in range(len(copies)):
        for ps in range(rm['passes']):
          _, _, cnt, nk, nb = rg.generate_unit(eng, il, rm, copies[cpy], region_[0], cpy, (seed * 7919 + k * 104729) & 0xFFFFFFFF,
                                               wl['sample'], 0, k, mode='philox', corrupt=corrupt, corrupt_seed=seed, fetch=False)
          if sample is not None:
            sample.take(eng.unit_read, (nb, nb), templates=cnt, te_kept=nk)
          pairs += cnt; nbytes += 2 * nb; k += 1
      for cp in copies:
        eng.free_copy(cp)
    return pairs, nbytes

  def barrier():
    torch.cuda.synchronize()
    if world > 1:
      dist.barrier()
      torch.cuda.synchronize()

  # ---- value: inputs resident in HBM, outputs stay in HBM
  rids = [eng.load_region(refs[wl['regions'][ci]], wl['regions'][ci][1]) for ci in mine]
  sample = None
  if args.dump_outputs:
    # the last timed step copies windows of each unit's output to page-locked memory on the library's copy stream,
    # next to the following unit's kernels: that step's outputs themselves are recorded, not a later rerun
    sample = OutputSample(args.dump_outputs, sum(len(vcf_df[ci]['v']) for ci in mine) * rm['passes'], eng.pinned)
  clocks = ClockSampler(local); clocks.start()
  for w in range(args.warmup):
    value_step(1000 + w, rids)
  barrier()
  eng.prof_reset()
  clocks.mark()
  ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  pairs = nbytes = 0
  with torch.cuda.stream(stream):
    ev0.record(stream)
    for s in range(args.steps):
      p_, b_ = value_step(2000 + s, rids, sample if s == args.steps - 1 else None)
      pairs += p_; nbytes += b_
    ev1.record(stream)
  barrier()
  ms = ev0.elapsed_time(ev1)
  if sample is not None:
    eng.wait_copies()
    sample.write()
  clk = clocks.stop()
  prof = eng.prof()
  for rid in rids:
    eng.free_region(rid)

  def allsum(x):
    if world == 1:
      return float(x)
    t = torch.tensor([float(x)], dtype=torch.float64, device='cuda')
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t[0])

  def allmax(x):
    if world == 1:
      return float(x)
    t = torch.tensor([float(x)], dtype=torch.float64, device='cuda')
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t[0])

  pairs_all, ms_max, nbytes_all = allsum(pairs), allmax(ms), allsum(nbytes)

  # ---- e2e: host buffers in, the product's worker + the native sink out
  e2e = None
  if not args.no_e2e:
    schedule = list(rg.get_data_for_workers(rm, vcf_df, args.seed))
    bytes_per_step = nbytes_all / max(1, args.steps)
    table = '/dev/shm/mitty_b200_bench_{}.tbl'.format(os.environ.get('MASTER_PORT', str(os.getpid()))) if world > 1 else None
    span = max(r[2] - r[1] for r in wl['regions'])
    chunk = max(1 << 16, min(rg.CHUNK_BYTES, int(span * 1.05 * rm['p'] * 1.2 * (2 * L + 150)) + (1 << 16)))
    n_writers = max(2, min(32, (os.cpu_count() or 8) // max(1, world)))

    def e2e_step(seed, p1, p2):
      sink = None
      if rank == 0:
        sink = Sink(p1, p2, len(schedule), n_producers=1, slots=rg.SLOTS_PER_GPU, chunk_bytes=chunk, threads=n_writers, table=table, owner=True)
      if world > 1:
        dist.barrier()                           # the table exists and the outputs are truncated
      if rank != 0:
        sink = Sink(p1, p2, len(schedule), n_producers=1, slots=rg.SLOTS_PER_GPU, chunk_bytes=chunk, threads=n_writers, table=table, owner=False)
      if world > 1:
        dist.barrier()
      t0 = time.perf_counter()
      n = rg.gpu_worker(local, 0, sink, schedule, vcf_df, fetch_ref, il, rm, wl['sample'], 'philox', corrupt, seed, engine=eng)
      w = sink.close()                           # every byte of this rank is written
      if world > 1:
        dist.barrier()
      return n, w[0] + w[1], time.perf_counter() - t0

    def e2e_leg(p1, p2, warm, steps):
      for w in range(warm):
        e2e_step(3000 + w, p1, p2)
      ep = eb = 0
      e_wall = 0.0
      for s in range(steps):
        n, wb, dt = e2e_step(4000 + s, p1, p2)
        ep += n; eb += wb; e_wall += dt
      for f in (p1, p2, table):
        if rank == 0 and f and f != '/dev/null' and os.path.exists(f):
          os.remove(f)
      return {'pairs': allsum(ep), 'wall': allmax(e_wall), 'bytes': allsum(eb), 'steps': steps}

    # primary: host buffers (the sink's page-locked slots), handed in schedule order to the writer threads, target
    # /dev/null -- the device-to-host side of the path, what `generate-reads ... >(consumer)` sees from the engine
    e_steps = args.e2e_steps if args.e2e_steps is not None else max(1, min(args.steps, int(120.0 / max(1e-3, bytes_per_step / 45e9))))
    _, _, null_desc = pick_sink(argparse.Namespace(sink='/dev/null'), bytes_per_step)
    e2e = e2e_leg('/dev/null', '/dev/null', min(args.warmup, 3), e_steps)
    h2d = sum(refs[r['region']].nbytes + sum(v.pos.nbytes + v.op.nbytes + v.oplen.nbytes + v.alt_pool.nbytes + v.alt_off.nbytes for v in r['v']) for r in vcf_df)
    e2e.update(h2d=h2d, sink=null_desc, writers=n_writers)
    # second figure: the same into real files on tmpfs, when a step's FASTQ fits there (and in RAM)
    f1, f2, file_desc = pick_sink(args, bytes_per_step)
    if f1 != '/dev/null':
      fs = e2e_leg(f1, f2, 1, max(1, min(3, e_steps)))
      e2e['file'] = {'value': fs['pairs'] / fs['wall'], 'unit': 'pairs/s', 'pairs_per_min': 60.0 * fs['pairs'] / fs['wall'], 'sink': file_desc,
                     'gbs_written': fs['bytes'] / fs['wall'] / 1e9, 'steps': fs['steps'], 'writer_threads_per_rank': n_writers}
    else:
      e2e['file'] = {'value': None, 'sink': 'not measured: one step ({:.0f} GB of FASTQ) does not fit /dev/shm + RAM of this box'.format(bytes_per_step / 1e9)}

    # the ceiling of e2e: N concurrent page-locked device-to-host streams, one per rank (tools/pcie_bw.py does the same stand-alone)
    nb = 1 << 30
    d = torch.empty(nb, dtype=torch.uint8, device='cuda')
    h = torch.empty(nb, dtype=torch.uint8).pin_memory()
    h.copy_(d, non_blocking=True); barrier()
    t0 = time.perf_counter()
    for _ in range(4):
      h.copy_(d, non_blocking=True)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if world > 1:
      dist.barrier()
    e2e['d2h_ceiling_gbs'] = allsum(4 * nb) / allmax(dt) / 1e9
    del d, h

  if rank == 0:
    peak, peak_src = measured_peak()
    # dominant kernel: k_unit_emit.  Algorithmic bytes per launch = FASTQ bytes written (both files)
    # + 2 * ceil(L/4) haplotype bytes read per pair (SURVEY.md 8d), over the CUDA-event time of the
    # emit launches (events recorded around each launch on the launch stream inside the library).
    alg = nbytes + pairs * 2 * ((L + 3) // 4)
    ach = alg / (prof['emit_ms'] * 1e-3) / 1e9 if prof['emit_ms'] > 0 else 0.0
    traffic = None
    tp = os.path.join(ROOT, 'profiles', 'traffic.json')   # dram bytes per launch of k_unit_emit from the committed ncu --set full capture
    if os.path.exists(tp) and args.workload == 'chr1':
      try:
        traffic = json.load(open(tp)).get('corrupt' if corrupt else 'perfect', {}).get(str(args.contig_len))
      except Exception:
        traffic = None
    value = pairs_all / (ms_max * 1e-3)
    line = {'metric': 'read pairs/sec (2x150, FASTQ-formatted, corrupted)' if corrupt else 'read pairs/sec (2x150, FASTQ-formatted, perfect reads)',
            'value': value, 'unit': 'pairs/s', 'pairs_per_min': 60.0 * value, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': ms_max / args.steps, 'higher_is_better': True, 'scaling': 'strong' if args.workload == 'wgs' else 'weak', 'vs_baseline': None,
            'dtype': 'u8', 'data': 'synthetic',
            'config': config_dict(args),          # the same dict on both arms (--impl reference prints it too)
            'host_binding': 'rank 0 on cores {}..{} (GPU-local, NVML)'.format(numa_cores[0], numa_cores[-1]) if numa_cores else 'none',
            'clocks': clk, 'gpu_launches': prof['total_launches'],
            'roofline': {'bound': 'hbm', 'kernel': 'k_unit_emit', 'achieved': ach, 'peak': peak, 'unit': 'GB/s', 'frac': ach / peak,
                         'traffic': traffic, 'peak_source': peak_src, 'launches': prof['emit_launches'],
                         'avg_launch_ms': prof['emit_ms'] / max(1, prof['emit_launches']),
                         'algorithmic_bytes_per_launch': alg / max(1, prof['emit_launches']),
                         'algorithmic_bytes_per_pair': alg / max(1, pairs),
                         'other_kernels': dict({'k_unit_plan_avg_ms': prof['plan_ms'] / max(1, prof['emit_launches'])}, **other_kernels())}}
    if e2e:
      ev = e2e['pairs'] / e2e['wall']
      line['e2e'] = {'value': ev, 'unit': 'pairs/s', 'pairs_per_min': 60.0 * ev, 'h2d_bytes_per_step': int(e2e['h2d']),
                     'd2h_bytes_per_step': int(e2e['bytes'] / max(1, e2e['steps'])), 'steps': e2e['steps'], 'sink': e2e['sink'],
                     'writer_threads_per_rank': e2e['writers'], 'gbs_written': e2e['bytes'] / e2e['wall'] / 1e9,
                     'd2h_ceiling_gbs': e2e['d2h_ceiling_gbs'], 'frac_of_d2h_ceiling': (e2e['bytes'] / e2e['wall'] / 1e9) / max(1e-9, e2e['d2h_ceiling_gbs']),
                     'file_sink': e2e['file'],
                     'host_inputs': 'page-locked' if pinned_keep else 'pageable', 'path': 'readgenerate.gpu_worker (units pulled in schedule order) -> drain thread (D2H) -> native sink'}
    if not args.no_cpu_baseline and world == 1:
      cwl = wl if args.workload == 'chr1' else {'contigs': [wl['contigs'][0]], 'tables': [wl['tables'][0]], 'sample': wl['sample']}
      n, wall, sl = port_baseline(cwl, 1)
      port = {'value': n / wall, 'unit': 'pairs/s', 'cores': 1, 'kind': 'port',
              'sample': 'one {} Mb-slice work unit of the same contig (generate + corrupt, {} pairs), C restatement of the reference, 1 thread'.format(sl // 1000000, n)}
      line['cpu_baseline'] = port
      if reference_available():
        try:
          T = max(1, min(os.cpu_count() or 1, 32))
          rr = ReferenceRunner(cwl, T)
          n, wall, tg, tc = rr.step(args.seed)
          rr.close()
          line['cpu_baseline'] = {'value': n / wall, 'unit': 'pairs/s', 'cores': T, 'nproc': os.cpu_count(), 'kind': 'reference',
                                  'sample': 'mitty generate-reads --threads {T} + mitty corrupt-reads --threads {T} (unmodified reference, baseline/_ref) on a {kb} kb slice, '
                                            '{n} pairs; generate {g:.0f} / corrupt {c:.0f} pairs/s'.format(T=T, kb=rr.slice // 1000, n=n, g=n / max(tg, 1e-9), c=n / max(tc, 1e-9)),
                                  'port': port}
        except Exception as e:  # noqa: B902 -- the port figure stands
          line['cpu_baseline']['reference_error'] = repr(e)[:200]
    emit(line)
  eng.close()
  if world > 1:
    dist.destroy_process_group()


def bench_corrupt_reads(args, eng, rm, model):
  """Standalone `corrupt-reads` (readcorrupt.multi_process's kernel path) over the perfect reads of one
  chr1-shaped unit: the kernel alone (CUDA events inside the library) against its 1480 B/pair roofline
  -- every FASTQ byte of both files read once and written once (SURVEY.md 8d) -- and through the C ABI
  with host buffers (H2D of the perfect reads, D2H of the corrupted ones)."""
  import mitty_b200.simulation.illumina as il
  from mitty_b200.engine import MODE_PHILOX
  from mitty_b200.lib import vcfio
  wl = make_chr1(args)
  region = wl['regions'][0]
  r = vcfio.from_variant_table(wl['tables'][0], region)
  rid = eng.load_region(np.ascontiguousarray(wl['contigs'][0][1]), region[1])
  cp = eng.build_copy(rid, r['v'][0])
  n = int((cp.p_max - cp.p_min) * rm['p'] * 1.2)
  f1, f2, cnt, _, nb = eng.generate_unit(cp, n, rm['p'], MODE_PHILOX, 4242, '@S:0:0:', '|1|0')
  eng.free_copy(cp); eng.free_region(rid)
  eng.load_model(model)
  chunk = 512 << 20
  p1, p2 = eng.pinned(chunk), eng.pinned(chunk)
  outs = (eng.pinned(chunk + (1 << 20)), eng.pinned(chunk + (1 << 20)))

  def one_pass(sample=None):
    """-> (templates, chunks) of one pass over the resident pair."""
    o1 = o2 = 0; done = 0; chunks = 0
    while o1 < f1.size:
      a1 = f1[o1:o1 + chunk]; a2 = f2[o2:o2 + chunk]
      p1[:a1.size] = a1; p2[:a2.size] = a2
      q1, q2, k, c1, c2 = eng.corrupt_fastq(p1[:a1.size], p2[:a2.size], mode=MODE_PHILOX, seed=args.seed, first_template=done, out=outs, partial=True)
      if sample is not None:
        sample.take(lambda m, off, n, dst: np.copyto(dst, (q1, q2)[m][off:off + n]), (q1.size, q2.size), templates=k)  # noqa: B023
      o1 += c1; o2 += c2; done += k; chunks += 1
    return done, chunks

  for _ in range(max(1, min(args.warmup, 2))):
    _, n_chunks = one_pass()
  # every pass cuts the same input into the same chunks: the warm-up's count is the count of the last timed pass
  sample = OutputSample(args.dump_outputs, n_chunks, eng.pinned) if args.dump_outputs else None
  eng.prof_reset()
  t0 = time.perf_counter()
  pairs = 0
  for s in range(args.steps):
    pairs += one_pass(sample if s == args.steps - 1 else None)[0]
  wall = time.perf_counter() - t0
  if sample is not None:
    sample.write()
  prof = eng.prof()
  peak, peak_src = measured_peak()
  alg = 2.0 * (f1.size + f2.size) * args.steps                          # read once + written once, both files
  ach = alg / (prof['emit_ms'] * 1e-3) / 1e9
  line = {'metric': 'read pairs/sec (2x150, corrupt-reads over resident FASTQ)', 'value': pairs / (prof['emit_ms'] * 1e-3), 'unit': 'pairs/s', 'n_gpus': 1,
          'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': prof['emit_ms'] / args.steps, 'higher_is_better': True, 'scaling': 'weak',
          'vs_baseline': None, 'dtype': 'u8', 'data': 'synthetic',
          'config': {'workload': 'corrupt-reads over the perfect reads of one chr1-shaped unit ({} pairs, 2 x {:.2f} GB), Philox mode, 512 MB chunks'.format(cnt, f1.size / 1e9)},
          'gpu_launches': prof['total_launches'],
          'roofline': {'bound': 'hbm', 'kernel': 'k_corrupt_staged', 'achieved': ach, 'peak': peak, 'unit': 'GB/s', 'frac': ach / peak, 'traffic': None,
                       'peak_source': peak_src, 'launches': prof['emit_launches'], 'avg_launch_ms': prof['emit_ms'] / max(1, prof['emit_launches']),
                       'algorithmic_bytes_per_pair': alg / max(1, pairs)},
          'e2e': {'value': pairs / wall, 'unit': 'pairs/s', 'h2d_bytes_per_step': int(f1.size + f2.size), 'd2h_bytes_per_step': int(f1.size + f2.size),
                  'sink': 'pinned host memory (mg_corrupt_fastq with host buffers; includes the host-side staging memcpy of this script)'}}
  emit(line)
  eng.close()


def other_kernels():
  """Second-figure rooflines measured by other invocations of this round (profiles/other_kernels.json)."""
  p = os.path.join(ROOT, 'profiles', 'other_kernels.json')
  if os.path.exists(p):
    try:
      return json.load(open(p))
    except Exception:
      pass
  return {}


if __name__ == '__main__':
  main()
