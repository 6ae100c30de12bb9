"""ctypes binding of libmitty_b200.so (include/mitty_b200.h).

The library is built in-tree by ``build()`` (nvcc, sm_100a only) and loaded from
``mitty_b200/libmitty_b200.so``.  There is no CPU fallback: if the library is missing, or there is
no CUDA device, the first use raises.
"""
import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, 'csrc')
SO_PATH = os.path.join(_HERE, 'libmitty_b200.so')
SOURCES = ['mg_api.cu', 'mg_kernels.cu', 'mg_check.cu', 'mg_bam.cu', 'mg_readmodel.cu', 'mg_sink.cpp', 'mg_bgzf.cpp', 'mg_fasta.cpp']
HEADERS = ['mg_core.cuh', 'mg_internal.h', 'mg_qname.cuh', 'mg_bgzf.h', 'mg_deflate.h', 'mg_sink.cpp', 'mg_check.cu', 'mg_fasta.cpp', os.path.join('..', '..', 'include', 'mitty_b200.h')]
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC', '-shared', '-lz']

MG_OK, MG_ECUDA, MG_EINVAL, MG_ECAP, MG_EVALUE, MG_EINDEX = 0, -1, -2, -3, -4, -5
MODE_PHILOX, MODE_DET, MODE_EXPLICIT = 0, 1, 2

# every symbol include/mitty_b200.h declares
SYMBOLS = ['mg_device_count', 'mg_ctx_create', 'mg_ctx_destroy', 'mg_last_error', 'mg_synchronize', 'mg_host_alloc', 'mg_host_free', 'mg_model_load', 'mg_model_tables',
           'mg_region_load', 'mg_region_free', 'mg_copy_build', 'mg_copy_free', 'mg_copy_nodes',
           'mg_copy_haplotype', 'mg_sample_templates', 'mg_unit_generate', 'mg_unit_generate_async', 'mg_wait_copies', 'mg_unit_read_async', 'mg_corrupt_fastq',
           'mg_prof_reset', 'mg_prof_get', 'mg_sink_create', 'mg_sink_create_shared', 'mg_sink_next_unit', 'mg_sink_unit_size', 'mg_sink_acquire', 'mg_sink_commit', 'mg_sink_abort',
           'mg_sink_commit_multi', 'mg_sink_prealloc', 'mg_sink_error', 'mg_sink_chunk_bytes', 'mg_sink_close', 'mg_unit_drain_async', 'mg_drain_wait',
           'mg_batch_build', 'mg_batch_free', 'mg_batch_generate',
           'mg_fasta_open', 'mg_fasta_close', 'mg_fasta_n_contigs', 'mg_fasta_contig', 'mg_fasta_fetch',
           'mg_check_open', 'mg_check_close', 'mg_check_add_copy', 'mg_check_fastq',
           'mg_bam_open', 'mg_bam_add', 'mg_bam_close', 'mg_bam_abort', 'mg_bam_write_sorted',
           'mg_bam_scan', 'mg_readmodel_bam']


class UnitDesc(C.Structure):
  _fields_ = [('copy_id', C.c_int64), ('n_candidates', C.c_int64), ('p', C.c_double), ('mode', C.c_int32),
              ('unit_seed', C.c_uint32), ('ts', C.c_void_p), ('u_tlen', C.c_void_p), ('tl', C.c_void_p),
              ('fo', C.c_void_p), ('qname_prefix', C.c_char_p), ('qname_mid', C.c_char_p),
              ('corrupt', C.c_int32), ('corrupt_seed', C.c_uint32), ('p_min', C.c_int64), ('p_max', C.c_int64)]


def needs_build():
  if not os.path.exists(SO_PATH):
    return True
  t = os.path.getmtime(SO_PATH)
  return any(os.path.getmtime(os.path.join(_CSRC, f)) > t for f in SOURCES + HEADERS)


def build(force=False, verbose=False):
  """Compile the CUDA library for sm_100a (cross-compiles without a GPU)."""
  if not force and not needs_build():
    return SO_PATH
  cmd = ['nvcc'] + NVCC_FLAGS + (['-Xptxas', '-v'] if verbose else []) + ['-o', SO_PATH] + SOURCES
  subprocess.check_call(cmd, cwd=_CSRC)
  return SO_PATH


_lib = None


def lib():
  global _lib
  if _lib is None:
    if not os.path.exists(SO_PATH):
      raise RuntimeError('mitty_b200: {} is missing. Build it with `python -c "import __graft_entry__ as g; g.build()"` '
                         '(needs nvcc). There is no CPU fallback.'.format(SO_PATH))
    L = C.CDLL(SO_PATH)
    for name in SYMBOLS:
      getattr(L, name)  # AttributeError here means header and library disagree
    L.mg_last_error.restype = C.c_char_p
    L.mg_last_error.argtypes = [C.c_void_p]
    L.mg_ctx_destroy.restype = None
    L.mg_ctx_destroy.argtypes = [C.c_void_p]
    L.mg_ctx_create.argtypes = [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]
    L.mg_synchronize.argtypes = [C.c_void_p]
    L.mg_host_alloc.argtypes = [C.c_void_p, C.c_int64, C.POINTER(C.c_void_p)]
    L.mg_host_free.argtypes = [C.c_void_p, C.c_void_p]
    L.mg_model_load.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int]
    L.mg_model_tables.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    L.mg_region_load.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.POINTER(C.c_int64)]
    L.mg_region_free.argtypes = [C.c_void_p, C.c_int64]
    L.mg_copy_build.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    L.mg_copy_free.argtypes = [C.c_void_p, C.c_int64]
    L.mg_copy_nodes.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.mg_copy_haplotype.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64]
    L.mg_sample_templates.argtypes = [C.c_void_p, C.POINTER(UnitDesc), C.c_void_p, C.c_void_p, C.c_void_p]
    L.mg_unit_generate.argtypes = [C.c_void_p, C.POINTER(UnitDesc), C.c_void_p, C.c_void_p, C.c_int64,
                                   C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    L.mg_unit_generate_async.argtypes = L.mg_unit_generate.argtypes
    L.mg_wait_copies.argtypes = [C.c_void_p]
    L.mg_unit_read_async.argtypes = [C.c_void_p, C.c_int32, C.c_int64, C.c_int64, C.c_void_p]
    L.mg_corrupt_fastq.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int32, C.c_uint32,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                   C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.c_int64,
                                   C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    L.mg_prof_reset.argtypes = [C.c_void_p]
    L.mg_prof_get.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_double)]
    L.mg_sink_create.argtypes = [C.c_char_p, C.c_char_p, C.c_int64, C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.POINTER(C.c_void_p)]
    L.mg_sink_create_shared.argtypes = [C.c_char_p, C.c_char_p, C.c_int64, C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_char_p, C.c_int32, C.POINTER(C.c_void_p)]
    L.mg_sink_next_unit.argtypes = [C.c_void_p]
    L.mg_sink_next_unit.restype = C.c_int64
    L.mg_sink_unit_size.argtypes = [C.c_void_p, C.c_int64, C.c_int64]
    L.mg_sink_acquire.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]
    L.mg_sink_commit.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64]
    L.mg_sink_commit_multi.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.mg_batch_build.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int64), C.c_void_p, C.c_void_p]
    L.mg_batch_free.argtypes = [C.c_void_p, C.c_int64]
    L.mg_batch_generate.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_char_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_double, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                    C.c_uint32, C.c_void_p, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.c_void_p, C.c_void_p]
    L.mg_sink_prealloc.argtypes = [C.c_int64, C.c_int32, C.c_int32]
    L.mg_sink_prealloc.restype = C.c_int32
    L.mg_sink_abort.argtypes = [C.c_void_p, C.c_char_p]
    L.mg_sink_abort.restype = None
    L.mg_sink_error.argtypes = [C.c_void_p]
    L.mg_sink_error.restype = C.c_char_p
    L.mg_sink_chunk_bytes.argtypes = [C.c_void_p]
    L.mg_sink_chunk_bytes.restype = C.c_int64
    L.mg_sink_close.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    L.mg_unit_drain_async.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int64]
    L.mg_drain_wait.argtypes = [C.c_void_p]
    L.mg_fasta_open.argtypes = [C.c_char_p, C.POINTER(C.c_void_p)]
    L.mg_fasta_close.argtypes = [C.c_void_p]
    L.mg_fasta_close.restype = None
    L.mg_fasta_n_contigs.argtypes = [C.c_void_p]
    L.mg_fasta_n_contigs.restype = C.c_int64
    L.mg_fasta_contig.argtypes = [C.c_void_p, C.c_int64, C.POINTER(C.c_char_p), C.POINTER(C.c_int64), C.POINTER(C.c_int32)]
    L.mg_fasta_fetch.argtypes = [C.c_void_p, C.c_char_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int32]
    L.mg_fasta_fetch.restype = C.c_int64
    L.mg_check_open.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
    L.mg_check_close.argtypes = [C.c_void_p]
    L.mg_check_close.restype = None
    L.mg_check_add_copy.argtypes = [C.c_void_p, C.c_int64, C.c_char_p, C.c_int32]
    L.mg_check_fastq.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                                 C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    L.mg_bam_open.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_char_p, C.c_char_p, C.c_int32, C.c_int32,
                              C.c_int64, C.POINTER(C.c_void_p)]
    L.mg_bam_add.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                             C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int32)]
    L.mg_bam_close.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.c_void_p]
    L.mg_bam_abort.argtypes = [C.c_void_p]
    L.mg_bam_abort.restype = None
    L.mg_bam_write_sorted.argtypes = [C.c_char_p, C.c_char_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_char_p, C.c_void_p, C.c_int64, C.c_int32,
                                      C.c_int32, C.POINTER(C.c_int64)]
    L.mg_bam_scan.argtypes = [C.c_char_p, C.c_int32, C.c_int64, C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int32)]
    L.mg_readmodel_bam.argtypes = [C.c_void_p, C.c_char_p, C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int32)]
    _lib = L
  return _lib
