"""noise3 and the terrain octaves' arguments exactly where a different rounding or tie rule would show.

The device code picks noise3's simplex region and extra-vertex case with selects instead of the
published nested branches, and computes the octaves' `x / size` quotients with a reciprocal and an
exact-remainder correction instead of `/`.  Both must give the same doubles as the reference:

* on a 1/12 lattice every region test meets its ties exactly (in_sum in {1, 2}, xins == yins,
  p_k == 1, equal scores), and there the host-compiled noise3 must match the C oracle bit for bit and
  land in the case the published branches pick;
* every octave's arguments must equal the IEEE quotients for every coordinate a map side (< 32768)
  can produce.
"""
import ctypes
import math
import pathlib
import shutil
import subprocess

import numpy as np
import pytest

from oracle import build as oracle_build
from tests import hostsim_env


def _published_case(x, y, z):
  """Extra-vertex case id (numbering of cr_noise.h) chosen by the legacy OpenSimplex branches."""
  stretch = (x + y + z) * (-1.0 / 6.0)
  xs, ys, zs = x + stretch, y + stretch, z + stretch
  xins, yins, zins = xs - math.floor(xs), ys - math.floor(ys), zs - math.floor(zs)
  in_sum = xins + yins + zins
  bit = lambda c: c >> 1
  if in_sum <= 1:
    a_point, b_point, a_score, b_score = 0x01, 0x02, xins, yins
    if a_score >= b_score and zins > b_score:
      b_score, b_point = zins, 0x04
    elif a_score < b_score and zins > a_score:
      a_score, a_point = zins, 0x04
    wins = 1 - in_sum
    if wins > a_score or wins > b_score:
      return bit(b_point if b_score > a_score else a_point)
    return 3 + bit(7 ^ (a_point | b_point))
  if in_sum >= 2:
    a_point, b_point, a_score, b_score = 0x06, 0x05, xins, yins
    if a_score <= b_score and zins < b_score:
      b_score, b_point = zins, 0x03
    elif a_score > b_score and zins < a_score:
      a_score, a_point = zins, 0x03
    wins = 3 - in_sum
    if wins < a_score or wins < b_score:
      return 6 + bit(7 ^ (b_point if b_score < a_score else a_point))
    return 9 + bit(a_point & b_point)
  p1 = xins + yins
  a_score, a_point, a_far = (p1 - 1, 0x03, True) if p1 > 1 else (1 - p1, 0x04, False)
  p2 = xins + zins
  b_score, b_point, b_far = (p2 - 1, 0x05, True) if p2 > 1 else (1 - p2, 0x02, False)
  p3 = yins + zins
  score, point, far = (p3 - 1, 0x06, True) if p3 > 1 else (1 - p3, 0x01, False)
  if a_score <= b_score and a_score < score:
    a_point, a_far = point, far
  elif a_score > b_score and b_score < score:
    b_point, b_far = point, far
  if a_far == b_far:
    return 12 + bit(a_point & b_point) if a_far else 15 + bit(7 ^ (a_point | b_point))
  c1, c2 = (a_point, b_point) if a_far else (b_point, a_point)
  return 18 + 3 * bit(7 ^ c1) + bit(c2)


def test_noise3_on_region_boundaries_matches_oracle_and_published_branches():
  oracle = ctypes.CDLL(str(oracle_build.ensure()))
  oracle.osn_init.argtypes = [ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p]
  oracle.osn_noise3_array.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_int, ctypes.c_void_p]
  hs = hostsim_env.lib()
  hs.hs_noise3_case.argtypes = [ctypes.c_double] * 3
  perm, pgi = np.zeros(256, np.int16), np.zeros(256, np.int16)
  oracle.osn_init(4321, perm.ctypes.data, pgi.ctypes.data)
  perm8 = perm.astype(np.uint8)
  k = np.arange(-18, 19) / 12.0  # includes every multiple of 1/6 in [-1.5, 1.5]
  pts = np.stack(np.meshgrid(k, k, k, indexing='ij'), -1).reshape(-1, 3)
  pts = np.concatenate([pts, pts + np.array([3.0, -7.0, 11.0])])  # the same ties in other cells
  want = np.zeros(len(pts))
  oracle.osn_noise3_array(perm.ctypes.data, pgi.ctypes.data, np.ascontiguousarray(pts).ctypes.data, len(pts),
                          want.ctypes.data)
  cases = set()
  for (x, y, z), w in zip(pts.tolist(), want.tolist()):
    got = hs.hs_noise3(perm8.ctypes.data, x, y, z)
    assert got == w, (x, y, z, got, w)
    case = hs.hs_noise3_case(x, y, z)
    assert case == _published_case(x, y, z), (x, y, z, case)
    cases.add(case)
  assert cases == set(range(27)) - {18, 22, 26}


# octave index (wg_octave_code) -> (x numerator factor, x divisors, y factor, y divisors, z); worldgen.py:27-60
OCTAVES = {
    0: (1, [15], 1, [15], 3), 1: (1, [5], 1, [5], 3), 2: (1, [15], 1, [15], 0), 3: (1, [5], 1, [5], 0),  # water, mountain
    4: (1, [3], 1, [3], 8),                                                       # start
    8: (1, [7], 1, [7], 6), 12: (1, [9], 1, [9], 4), 16: (1, [7], 1, [7], 5),      # cave, sand, tree
    20: (2, [3], 1, [5, 3], 7), 21: (1, [5, 3], 2, [3], 7),                        # tunnels (2x, y/5) / (x/5, 2y) over 3
    22: (1, [8], 1, [8], 1), 23: (1, [6], 1, [6], 2),                              # coal, iron
    24: (1, [5], 1, [5], 6),                                                      # lava
}


CSRC = pathlib.Path(__file__).resolve().parents[1] / 'crafter_b200' / 'csrc'

# noise3's arguments of octave `index` (wg_octave_code's numbering) at x = y = v, v = 0 .. n - 1, through the
# functions k_wg_mat stages (wg_octave) and calls per item (wg_octave_args); compiled for the host like tests/hostsim
OCTAVE_ARGS_SRC = r"""
#define CR_HOSTSIM 1
#include "cr_common.h"
#include "cr_worldgen.h"
using namespace cr;
extern "C" void octave_args(int index, int n, double *ax, double *ay, double *az) {
  const WgOctave o = wg_octave(wg_octave_code(index));
  for (int v = 0; v < n; ++v) wg_octave_args(o, v, v, ax[v], ay[v], az[v]);
}
"""


@pytest.fixture(scope='module')
def octave_args(tmp_path_factory):
  if shutil.which('g++') is None:
    pytest.skip('no g++')
  d = tmp_path_factory.mktemp('octave_args')
  (d / 'octave_args.cpp').write_text(OCTAVE_ARGS_SRC)
  subprocess.run(['g++', '-O2', '-std=c++17', '-ffp-contract=off', '-fno-fast-math', '-fPIC', '-shared',
                  '-I', str(CSRC), '-o', str(d / 'liboctave_args.so'), str(d / 'octave_args.cpp'), '-lm'], check=True)
  lib = ctypes.CDLL(str(d / 'liboctave_args.so'))
  lib.octave_args.argtypes = [ctypes.c_int, ctypes.c_int] + [ctypes.c_void_p] * 3
  return lib.octave_args


def test_octave_arguments_are_the_ieee_quotients_for_every_map_coordinate(octave_args):
  n = 32768
  v = np.arange(n, dtype=np.float64)
  for index, (mx, dx, my, dy, z) in OCTAVES.items():
    ax, ay, az = np.zeros(n), np.zeros(n), np.zeros(n)
    octave_args(index, n, ax.ctypes.data, ay.ctypes.data, az.ctypes.data)
    wx, wy = mx * v, my * v
    for d in dx:
      wx = wx / d
    for d in dy:
      wy = wy / d
    assert np.array_equal(ax, wx), (index, np.flatnonzero(ax != wx)[:5])
    assert np.array_equal(ay, wy), (index, np.flatnonzero(ay != wy)[:5])
    assert (az == z).all(), index
