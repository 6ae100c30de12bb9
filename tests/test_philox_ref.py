"""CPU checks of the numpy specification's header rule (tests/philox_ref.py): the standalone corrupt-reads
heads both output files with '@' + read 1's name, cut at the first space, tab or CR."""
import numpy as np

from tests import philox_ref as PR


def _tables():
  """Two mates x 8 cycles of alias rows whose every entry means quality 30, no substitution."""
  alias = np.full((2, 8, 32), (0xFFFF << 16) | (30 << 8) | 30, dtype=np.uint32)
  return alias, 5, 0


def test_record_name():
  assert PR.record_name(b'@read1') == b'read1'
  assert PR.record_name(b'@read1 comment with spaces') == b'read1'
  assert PR.record_name(b'@r\tx y') == b'r'
  assert PR.record_name(b'@r\rx') == b'r'
  assert PR.record_name(b'@') == b''
  assert PR.record_name(b'@ leading') == b''
  assert PR.record_name(b'>r|x:y') == b'r|x:y'       # only space, tab and CR end a name


def test_names_from_replaces_only_the_header_lines():
  fq1 = b'@a1 c1\nACGT\n+\nIIII\n@a2\tc2\nAC\n+\nII\n@\nA\n+\nI\n'
  fq2 = b'@b1\nTTTTT\n+\nIIIII\n@b2 x\nGG\n+\nII\n@b3\nC\n+\nI\n'
  tabs = _tables()
  own2 = PR.corrupt_file(fq2, 1, tabs, 7, 9)
  got2 = PR.corrupt_file(fq2, 1, tabs, 7, 9, names_from=fq1)
  assert own2.split(b'\n')[0::4] == [b'@b1', b'@b2 x', b'@b3', b'']
  assert got2.split(b'\n')[0::4] == [b'@a1', b'@a2', b'@', b'']
  for k in (1, 2, 3):            # sequence, '+' and quality lines are untouched by the header rule
    assert got2.split(b'\n')[k::4] == own2.split(b'\n')[k::4]
  assert own2.split(b'\n')[3::4][:3] == [b'?????', b'??', b'?']        # quality 30 everywhere
  # file 1 with its own names: the comment goes, as in the kernel
  assert PR.corrupt_file(fq1, 0, tabs, 7, 9, names_from=fq1).split(b'\n')[0::4] == [b'@a1', b'@a2', b'@', b'']
