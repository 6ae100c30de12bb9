"""The decimal digit counts of mitty_b200/csrc/mg_core.cuh (mg_ndigits_ones, mg_ndigits32, mg_nchars_i32,
mg_ndigits, mg_digit_sum), compiled with g++ and checked against Python's str().  Every record size and byte
offset of a unit goes through them: the CIGAR / POS / v_list numbers and the serial in the qname."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
HEADER = os.path.join(HERE, '..', 'mitty_b200', 'csrc', 'mg_core.cuh')

SHIM = r'''
#include "%s"
extern "C" {
void nd_ones(const uint32_t *v, int64_t n, int32_t *d, uint32_t *ones) {
  for (int64_t i = 0; i < n; i++) { uint32_t o; d[i] = mg_ndigits_ones(v[i], o); ones[i] = o; }
}
void nd32(const uint32_t *v, int64_t n, int32_t *d) { for (int64_t i = 0; i < n; i++) d[i] = mg_ndigits32(v[i]); }
void nchars(const int32_t *v, int64_t n, int32_t *d) { for (int64_t i = 0; i < n; i++) d[i] = mg_nchars_i32(v[i]); }
void nd64(const uint64_t *v, int64_t n, int32_t *d) { for (int64_t i = 0; i < n; i++) d[i] = mg_ndigits(v[i]); }
void dsum(const uint64_t *v, int64_t n, uint64_t *s) { for (int64_t i = 0; i < n; i++) s[i] = mg_digit_sum(v[i]); }
}
'''


@pytest.fixture(scope='module')
def shim(tmp_path_factory):
  d = tmp_path_factory.mktemp('digits')
  src, so = d / 'digits.cpp', d / 'libdigits.so'
  src.write_text(SHIM % os.path.abspath(HEADER))
  subprocess.check_call(['g++', '-O2', '-std=c++17', '-shared', '-fPIC', '-x', 'c++', str(src), '-o', str(so)])
  return C.CDLL(str(so))


def ptr(a):
  return a.ctypes.data_as(C.c_void_p)


def run(lib, name, v, out_dtype, n_out=1):
  outs = [np.zeros(v.size, dtype=out_dtype if isinstance(out_dtype, type) else out_dtype[i]) for i in range(n_out)]
  getattr(lib, name)(ptr(v), C.c_int64(v.size), *[ptr(o) for o in outs])
  return outs


def want_digits(v):
  """Decimal digits of each (non-negative) value, from Python's str()."""
  return np.array([len(str(int(x))) for x in v], dtype=np.int32)


def boundaries32():
  v = [0, 1, 2, 2 ** 31 - 1, 2 ** 31, 2 ** 32 - 2, 2 ** 32 - 1]
  for k in range(1, 10):
    v += [10 ** k - 1, 10 ** k, 10 ** k + 1]
  for b in range(1, 33):      # both ends of every bit length
    v += [2 ** (b - 1), 2 ** b - 1]
  return np.array(sorted(set(v)), dtype=np.uint32)


def random32(n, seed):
  """n values spread over every bit length (uniform values would almost all have ten digits)."""
  rng = np.random.default_rng(seed)
  return (rng.integers(0, 2 ** 32, n, dtype=np.uint64) >> rng.integers(0, 32, n, dtype=np.uint64)).astype(np.uint32)


def test_ndigits_ones_boundaries(shim):
  v = boundaries32()
  d, ones = run(shim, 'nd_ones', v, (np.int32, np.uint32), 2)
  want = want_digits(v)
  assert (d == want).all()
  assert (ones == np.array([int('1' * k) for k in want], dtype=np.uint32)).all()
  assert (run(shim, 'nd32', v, np.int32)[0] == want).all()


def test_ndigits_ones_random(shim):
  v = random32(3_000_000, 11)
  d, ones = run(shim, 'nd_ones', v, (np.int32, np.uint32), 2)
  # str() over three million values is slow; the digits follow from exact comparisons with the powers of ten
  want = 1 + sum((v.astype(np.uint64) >= 10 ** k).astype(np.int32) for k in range(1, 10))
  assert (d == want).all()
  assert (ones == np.array([(10 ** k - 1) // 9 for k in range(11)], dtype=np.uint64)[want].astype(np.uint32)).all()
  sub = v[:20000]
  assert (d[:20000] == want_digits(sub)).all()


def test_nchars_i32(shim):
  b = boundaries32().astype(np.int64)
  v = np.concatenate([b[b < 2 ** 31], -b[b <= 2 ** 31], random32(1_000_000, 12).astype(np.int64) - 2 ** 31])
  v = v.astype(np.int32)
  got = run(shim, 'nchars', v, np.int32)[0]
  assert (got[:4000] == np.array([len(str(int(x))) for x in v[:4000]], dtype=np.int32)).all()
  a = np.abs(v.astype(np.int64))
  want = (v < 0).astype(np.int32) + 1 + sum((a >= 10 ** k).astype(np.int32) for k in range(1, 10))
  assert (got == want).all()
  assert run(shim, 'nchars', np.array([-2 ** 31, 2 ** 31 - 1, -1, 0], dtype=np.int32), np.int32)[0].tolist() == [11, 10, 2, 1]


def test_ndigits64_and_digit_sum(shim):
  v = [0, 1, 9, 10, 2 ** 32 - 1, 2 ** 32, 2 ** 63, 2 ** 64 - 1]
  for k in range(1, 20):
    v += [10 ** k - 1, 10 ** k, 10 ** k + 1]
  v = np.array(sorted(set(v)), dtype=np.uint64)
  assert (run(shim, 'nd64', v, np.int32)[0] == want_digits(v)).all()
  # sum of the digits of 1..m, by blocks of equal length
  m = np.array([x for x in v.tolist() if x < 10 ** 17] + random32(2000, 13).tolist(), dtype=np.uint64)
  s = run(shim, 'dsum', m, np.uint64)[0]
  want = [sum((min(x, 10 ** d - 1) - 10 ** (d - 1) + 1) * d for d in range(1, len(str(x)) + 1)) if x else 0 for x in m.tolist()]
  assert s.tolist() == want
