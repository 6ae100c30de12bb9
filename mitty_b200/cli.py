"""Command line with the reference's ``generate-reads`` / ``corrupt-reads`` / ``qname`` commands
(mitty/cli.py:106-157), ``god-aligner`` (mitty/cli.py:191-204) and ``create-read-model bam2illumina``: same positional arguments and options, plus ``--deterministic`` (consume
the reference's numpy draws; byte-exact against ``mitty ... --threads 1``) and, for
generate-reads, ``--corrupt`` (fuse the corruption model into the emit kernel)."""
import logging
import os

import click

from mitty_b200.readmodels import builtin_models, get_read_model, load_model


@click.group()
@click.version_option()
@click.option('-v', '--verbose', type=int, default=0)
def cli(verbose):
  """B200-native engine for Mitty's read generation and corruption"""
  logging.basicConfig(level=[logging.ERROR, logging.WARNING, logging.INFO, logging.DEBUG][min(verbose, 3)])


@cli.command('filter-variants', short_help='Remove complex variants from VCF')
@click.argument('vcfin', type=click.Path(exists=True))
@click.argument('sample')
@click.argument('bed')
@click.argument('vcfout', type=click.Path())
def filter_vcf(vcfin, sample, bed, vcfout):
  """Subset VCF for given sample, apply BED file and filter out complex variants
   making it suitable to use for read generation (cli.py:20-29 of the reference)"""
  import mitty_b200.lib.vcfio as mvio
  mvio.prepare_variant_file(vcfin, sample, bed, vcfout)


@cli.command('list-read-models')
@click.option('-d', type=click.Path(exists=True), help='List models in this directory')
def list_read_models(d):
  """List read models"""
  import glob
  names = builtin_models() if d is None else glob.glob(os.path.join(d, '*'))
  for name in names:
    try:
      mod_data = load_model(name)
      click.echo('\n----------\n{}:\n{}\n=========='.format(os.path.basename(name), mod_data['model_description']))
    except Exception:
      logging.debug('Skipping {}. Not a read model file'.format(name))


@cli.command()
def qname():
  """Display qname format"""
  import mitty_b200.simulation.readgenerate as reads
  click.echo(reads.__qname_format_details__)


def print_qname(ctx, param, value):
  import mitty_b200.simulation.readgenerate as reads
  if not value or ctx.resilient_parsing:
    return
  click.echo(reads.__qname_format_details__)
  ctx.exit()


@cli.command('generate-reads', short_help='Generate simulated reads.')
@click.argument('fasta')
@click.argument('vcf')
@click.argument('sample_name')
@click.argument('bed')
@click.argument('modelfile')
@click.argument('coverage', type=float)
@click.argument('seed', type=int)
@click.argument('fastq1', type=click.Path())
@click.option('--fastq2', type=click.Path())
@click.option('--threads', default=2)
@click.option('--qname', is_flag=True, callback=print_qname, expose_value=False, is_eager=True, help='Print documentation for information encoded in qname')
@click.option('--deterministic', is_flag=True, help="Consume the reference's numpy draws: byte-exact vs `mitty generate-reads --threads 1`")
@click.option('--corrupt', is_flag=True, help='Fuse the Illumina corruption model into read generation (Philox draws)')
@click.option('--devices', default=None, help='comma separated CUDA devices (default: the first --threads GPUs)')
@click.option('--gzip', 'gzip_level', type=click.IntRange(0, 9), default=None, help='Write multi-member gzip at this level (default: 1 when FASTQ1 ends in .gz, else plain)')
@click.option('--workers-per-gpu', type=int, default=None, help='Host threads (own context and stream) per GPU (default 1)')
@click.option('--drop-end-deletions', is_flag=True, help='Leave out deletions that reach beyond the end of their BED region (default: error; the reference mis-handles them)')
def generate_reads(fasta, vcf, sample_name, bed, modelfile, coverage, seed, fastq1, fastq2, threads, deterministic, corrupt, devices, drop_end_deletions, gzip_level, workers_per_gpu):
  """Generate simulated reads (--threads = number of GPUs to use)"""
  import mitty_b200.simulation.readgenerate as reads
  if deterministic and corrupt:
    raise click.UsageError('--corrupt draws from Philox; for --deterministic run generate-reads and then corrupt-reads, as the reference does')
  read_module, model = get_read_model(modelfile)
  reads.process_multi_threaded(
    fasta, vcf, sample_name, bed, read_module, model, coverage,
    fastq1, fastq2, threads=threads, seed=seed,
    mode='deterministic' if deterministic else 'philox', corrupt=corrupt,
    devices=[int(x) for x in devices.split(',')] if devices else None, drop_end_deletions=drop_end_deletions, gzip_level=gzip_level, workers_per_gpu=workers_per_gpu)


@cli.command('check-reads', short_help='Verify that every read re-derives from its qname (god-aligner contract)')
@click.argument('fasta')
@click.argument('vcf')
@click.argument('sample_name')
@click.argument('bed')
@click.argument('fastq1', type=click.Path(exists=True))
@click.option('--fastq2', type=click.Path(exists=True))
@click.option('--device', default=0, help='CUDA device')
@click.option('--max-report', default=20, help='how many failing reads to print')
@click.option('--drop-end-deletions', is_flag=True, help='as given to generate-reads')
def check_reads(fasta, vcf, sample_name, bed, fastq1, fastq2, device, max_report, drop_end_deletions):
  """Re-derive every read of a FASTQ (pair) of PERFECT reads from its qname -- chrom, copy, strand,
  POS, CIGAR -- plus FASTA / VCF / BED, the way `mitty god-aligner` trusts it, and compare it with
  the bases in the file.  Exit status 1 if any read fails."""
  import mitty_b200.simulation.readcheck as chk
  res = chk.check_fastq(fasta, vcf, sample_name, bed, fastq1, fastq2, device=device, max_report=max_report, drop_end_deletions=drop_end_deletions)
  for f, rec, why, qname in res['examples']:
    click.echo('file {} record {}: {}: {}'.format(f, rec, why, qname))
  click.echo('{} reads of {} templates checked in {:0.2f}s: {} failed'.format(res['reads'], res['templates'], res['seconds'], res['bad']))
  if res['bad']:
    raise SystemExit(1)


@cli.command('god-aligner', short_help='Write the perfect alignments of simulated reads as a sorted, indexed BAM')
@click.argument('fasta', type=click.Path(exists=True))
@click.argument('fastq1', type=click.Path(exists=True))
@click.argument('bam', type=click.Path())
@click.option('--fastq2', type=click.Path(exists=True))
@click.option('--threads', type=int, default=None, help='host deflate threads (default: the cores of the box)')
@click.option('--device', default=0, help='CUDA device')
@click.option('--level', type=click.IntRange(0, 9), default=6, help='BGZF deflate level (0: stored blocks)')
def god_aligner(fasta, fastq1, bam, fastq2, threads, device, level):
  """Place every read exactly where its qname says: a coordinate-sorted BAM (and BAM.bai) of the
  perfect alignments, the truth set for an aligner or variant caller benchmark."""
  import mitty_b200.benchmarking.god_aligner as ga
  res = ga.process_multi_threaded(fasta, bam, fastq1, fastq2, threads=threads, device=device, level=level)
  click.echo('{} records written to {} in {:0.2f}s'.format(res['records'], bam, res['seconds']))


@cli.group('create-read-model')
def create_read_model():
  """Create a read model from data"""


@create_read_model.command('bam2illumina', short_help='Create an Illumina read model from a BAM')
@click.argument('bam', type=click.Path(exists=True))
@click.argument('pkl', type=click.Path())
@click.argument('description')
@click.option('--every', type=click.IntRange(1, (1 << 32) - 1), default=1, help='Count only every Nth record (file order)')
@click.option('--min-mq', type=click.IntRange(0), default=0, help='Skip reads with a lower mapping quality')
@click.option('--threads', type=int, default=None, help='host inflate threads (default: the cores of the box)')
@click.option('--max-bp', type=click.IntRange(1, 50000), default=300, help='Longest read counted (longer ones are skipped)')
@click.option('--max-tlen', type=click.IntRange(1, 1 << 20), default=1000, help='Template lengths at or above this are not counted')
@click.option('--device', default=0, help='CUDA device')
def bam2illumina(bam, pkl, description, every, min_mq, threads, max_bp, max_tlen, device):
  """Count base qualities per (mate, cycle), read lengths and template lengths of the alignments of BAM
  (a BGZF file or FIFO, any sort order) and write them as an Illumina read model PKL for generate-reads and
  corrupt-reads."""
  import mitty_b200.empirical.bam2illumina as b2i
  res = b2i.process_bam_parallel(bam, pkl, description, every=every, min_mq=min_mq, threads=threads, max_bp=max_bp, max_tlen=max_tlen,
                                 device=device)
  skipped = ', '.join('{} {}'.format(res['skip_' + k], why) for k, why in (
    ('flag', 'unmapped / secondary / QC-fail / supplementary'), ('mapq', 'below --min-mq'), ('empty', 'without SEQ'),
    ('noqual', 'without QUAL'), ('long', 'longer than --max-bp')))
  click.echo('{} of {} records counted ({} considered) in {:0.2f}s; skipped: {}'.format(
    res['counted'], res['records'], res['considered'], res['seconds'], skipped))


@cli.command('corrupt-reads', short_help='Apply corruption model to FASTQ file of reads')
@click.argument('modelfile')
@click.argument('fastq1_in', type=click.Path(exists=True))
@click.argument('fastq1_out', type=click.Path())
@click.argument('seed', type=int)
@click.option('--fastq2-in', type=click.Path(exists=True))
@click.option('--fastq2-out', type=click.Path())
@click.option('--threads', default=2)
@click.option('--deterministic', is_flag=True, help="Consume the reference's numpy draws: byte-exact vs `mitty corrupt-reads --threads 1`")
@click.option('--device', default=0, help='CUDA device')
def read_corruption(modelfile, fastq1_in, fastq1_out, seed, fastq2_in, fastq2_out, threads, deterministic, device):
  """Apply corruption model to FASTQ file of reads"""
  import mitty_b200.simulation.readcorrupt as rc
  read_module, read_model = get_read_model(modelfile)
  rc.multi_process(read_module, read_model, fastq1_in, fastq1_out, fastq2_in, fastq2_out, processes=threads, seed=seed,
                   mode='deterministic' if deterministic else 'philox', device=device)


if __name__ == '__main__':
  cli()
