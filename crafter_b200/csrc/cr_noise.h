// OpenSimplex (legacy, K. Spencer 2014) 3-D noise in IEEE double, the arithmetic the reference
// reaches through the un-vendored PyPI module `opensimplex` (worldgen.py:4,11,84-87; setup.py:16).
// Evaluated strictly left to right without FMA contraction (the translation unit is compiled with
// -fmad=false) so that thresholds on these doubles pick the same terrain as the CPU restatement.
// Tables (perm, perm_grad_index3, gradients) are staged in shared memory by the calling kernel.
#pragma once
#include "cr_common.h"

namespace cr {

constexpr int N_EXT_CASES = 27;

// World-independent tables, staged once per CTA (noise_const_init).  Everything noise3 needs as a double
// is READ as a double: int -> double conversions run at a quarter of the FP64 rate (profiles/, XU pipe).
struct NoiseConst {
  double grad[72];            // permutations of (+-11, +-4, +-4), as doubles
  double small[4];            // -1, 0, 1, 2
  double ksq[4];              // k * SQUISH, k = 0..3
  uint64_t ext[N_EXT_CASES];  // noise_ext_case(id), see noise3
};

struct NoiseTables {
  const uint8_t *perm;  // [256]
  const uint8_t *pgi;   // [256] (perm[i] % 24) * 3
  const NoiseConst *c;
};

// The 24 gradient vectors, in the order of the published table.
CR_DEV int8_t noise_gradient_component(int i) {
  // i = 3*g + c, g in 0..23.  Octant o = g / 3 carries signs (sx, sy, sz) with x flipping fastest;
  // within an octant the 11 moves through x, y, z.
  int g = i / 3, c = i - 3 * g;
  int o = g / 3, big = g - 3 * o;
  int sgn = c == 0 ? ((o & 1) ? 1 : -1) : (c == 1 ? ((o & 2) ? -1 : 1) : ((o & 4) ? -1 : 1));
  return (int8_t)(sgn * (c == big ? 11 : 4));
}

CR_DEV double noise_extrapolate(const NoiseTables &t, int xsb, int ysb, int zsb, double dx,
                                double dy, double dz) {
  int index = t.pgi[(t.perm[(t.perm[xsb & 0xFF] + ysb) & 0xFF] + zsb) & 0xFF];
  const double *gr = t.c->grad + index;
  return gr[0] * dx + gr[1] * dy + gr[2] * dz;
}

// One lattice contribution: attn = 2 - |d|^2, value += attn^4 * (gradient . d) when attn > 0.
// Evaluated unconditionally and committed by a select: the sum is the same double, but the ten
// table-lookup chains of a noise3 call carry no branches and overlap (out-of-range vertices only
// index the tables modulo 256).
#define CR_NOISE_CONTRIB(COND, XS, YS, ZS, DX, DY, DZ)                            \
  {                                                                               \
    const double attn_ = 2 - (DX) * (DX) - (DY) * (DY) - (DZ) * (DZ);             \
    const double e_ = noise_extrapolate(t, XS, YS, ZS, DX, DY, DZ);               \
    const double a2_ = attn_ * attn_;                                             \
    const double sum_ = value + a2_ * a2_ * e_;                                   \
    value = ((COND) && attn_ > 0) ? sum_ : value;                                 \
  }

// The published algorithm has three region blocks (tetrahedron at the origin, tetrahedron at
// (1,1,1), octahedron in between), each summing its own list of cube vertices and then two
// "extra" vertices.  Every cube vertex (i, j, k) uses the same displacement in all blocks,
//     d = (d0 - {i,j,k}) - (i + j + k) * SQUISH,
// and the blocks' lists are sub-sequences of  000, 100, 010, 001, 110, 101, 011, 111.  So all
// lanes walk that one sequence with a per-region membership mask: the same additions in the same
// order, but no divergence over the FP64-heavy part.
//
// The two extra vertices are chosen by nested branches on the in-cell coordinates; their leaves
// are 27 distinct assignments (N_EXT_CASES), each of the shape
//     lattice offset o,   displacement ((d0 - A) - k * SQUISH) - C      per axis, per extra vertex
// with A in {-1,0,1,2}, k in {0..3}, C in {0,1,2} and o = A + C (the published code writes e.g.
// `dy0 - 1 - 3*SQ` and later `-= 1`: A=1, k=3, C=1; subtracting a zero is exact).  A warp would
// otherwise execute the union of all leaves; here the region tests only pick a case number and the
// leaf is data: noise_ext_case(id) packs it into 6 bytes, staged once per CTA in shared memory.
// byte of (extra vertex e, axis a) at bits 8 * (3 * e + a): (A + 1) | k << 2 | C << 4
CR_DEV uint64_t noise_ext_pack(const int (&A)[2][3], const int (&K)[2][3], const int (&C)[2][3]) {
  uint64_t w = 0;
  for (int e = 0; e < 2; ++e)
    for (int a = 0; a < 3; ++a)
      w |= (uint64_t)((A[e][a] + 1) | (K[e][a] << 2) | (C[e][a] << 4)) << (8 * (3 * e + a));
  return w;
}

// Case numbering (c, c1, c2 are the published code's vertex bit sets; bit(c) = index of the single
// set bit, hole(c) = index of the single clear bit among the low three):
//    0.. 2  origin tetrahedron, one extra on a cube corner      id = bit(c)
//    3.. 5  origin tetrahedron, both on the far side             id = 3 + hole(c)
//    6.. 8  (1,1,1) tetrahedron, first sub-case                  id = 6 + hole(c)
//    9..11  (1,1,1) tetrahedron, second sub-case                 id = 9 + bit(c)
//   12..14  octahedron, both picks far                           id = 12 + bit(c)
//   15..17  octahedron, both picks near                          id = 15 + hole(c)
//   18..26  octahedron, one far (c1) one near (c2)               id = 18 + 3 * hole(c1) + bit(c2)
//           (18, 22, 26 -- hole(c1) == bit(c2) -- are never produced; tests/test_noise.py)
CR_DEV uint64_t noise_ext_case(int id) {
  int A[2][3] = {{0, 0, 0}, {0, 0, 0}}, K[2][3] = {{0, 0, 0}, {0, 0, 0}}, C[2][3] = {{0, 0, 0}, {0, 0, 0}};
  if (id < 3) {
    const int c = 1 << id;
    for (int a = 0; a < 3; ++a) {
      if (c & (1 << a)) { A[0][a] = A[1][a] = 1; }               // both on corner + 1: d0 - 1
      else if (a == 0) { A[0][a] = -1; A[1][a] = 0; }             // x: ext0 one back (d0 + 1), ext1 stays
      else if (a == 1) { if ((c & 1) == 0) A[1][a] = -1; else A[0][a] = -1; }
      else { A[0][a] = 0; A[1][a] = -1; }                         // z: ext1 one back
    }
  } else if (id < 6) {
    const int c = 7 ^ (1 << (id - 3));
    for (int a = 0; a < 3; ++a) {
      if (c & (1 << a)) { A[0][a] = A[1][a] = 1; K[0][a] = 2; K[1][a] = 1; }
      else { A[0][a] = 0; K[0][a] = 2; A[1][a] = -1; K[1][a] = 1; }
    }
  } else if (id < 9) {
    const int c = 7 ^ (1 << (id - 6));
    for (int a = 0; a < 3; ++a) {
      K[0][a] = K[1][a] = 3;
      if (a == 0) {
        if (c & 1) { A[0][a] = 2; A[1][a] = 1; }
      } else if (a == 1) {
        if (c & 2) { A[0][a] = A[1][a] = 1; if (c & 1) C[1][a] = 1; else C[0][a] = 1; }  // `-= 1` afterwards
      } else {
        if (c & 4) { A[0][a] = 1; A[1][a] = 2; }
      }
    }
  } else if (id < 12) {
    const int c = 1 << (id - 9);
    for (int a = 0; a < 3; ++a) {
      if (c & (1 << a)) { A[0][a] = 1; K[0][a] = 1; A[1][a] = 2; K[1][a] = 2; }
      else { K[0][a] = 1; K[1][a] = 2; }
    }
  } else if (id < 15) {
    const int big = id - 12;  // the axis of the single common bit
    for (int a = 0; a < 3; ++a) {
      A[0][a] = 1; K[0][a] = 3;
      K[1][a] = 2; A[1][a] = a == big ? 2 : 0;
    }
  } else if (id < 18) {
    const int back = id - 15;  // the axis missing from c
    for (int a = 0; a < 3; ++a) {
      K[1][a] = 1; A[1][a] = a == back ? -1 : 1;  // ext0 is the cell origin itself
    }
  } else {
    const int back = (id - 18) / 3, big = (id - 18) % 3;
    for (int a = 0; a < 3; ++a) {
      K[0][a] = 1; A[0][a] = a == back ? -1 : 1;
      K[1][a] = 2; C[1][a] = a == big ? 2 : 0;  // `d0 - 2*SQ`, then `-= 2`
    }
  }
  return noise_ext_pack(A, K, C);
}

CR_DEV int noise_bit(int c) { return c >> 1; }  // 1, 2, 4 -> 0, 1, 2

// Called by `nthreads` threads; the caller synchronises before the first noise3.
CR_DEV void noise_const_init(NoiseConst &c, int tid, int nthreads) {
  const double SQ = 1.0 / 3.0;
  for (int i = tid; i < 72; i += nthreads) c.grad[i] = (double)noise_gradient_component(i);
  for (int i = tid; i < 4; i += nthreads) { c.small[i] = (double)(i - 1); c.ksq[i] = (double)i * SQ; }
  for (int i = tid; i < N_EXT_CASES; i += nthreads) c.ext[i] = noise_ext_case(i);
}

CR_DEV double noise3(const NoiseTables &t, double x, double y, double z, int *case_out = nullptr) {
  const double SQ = 1.0 / 3.0;
  const double ST = -1.0 / 6.0;
  double stretch = (x + y + z) * ST;
  double xs = x + stretch, ys = y + stretch, zs = z + stretch;
  double fxs = floor(xs), fys = floor(ys), fzs = floor(zs);
  int xsb = (int)fxs, ysb = (int)fys, zsb = (int)fzs;
  // (the floors ARE the lattice coordinates as doubles: no int -> double conversions; sums of three
  // small integers are exact in either type)
  double squish = (fxs + fys + fzs) * SQ;
  double xb = fxs + squish, yb = fys + squish, zb = fzs + squish;
  double xins = xs - fxs, yins = ys - fys, zins = zs - fzs;
  double in_sum = xins + yins + zins;
  const double dx0 = x - xb, dy0 = y - yb, dz0 = z - zb;

  unsigned member;  // bit v set: cube vertex v of the sequence above contributes
  int id;           // which of the 27 extra-vertex assignments
  // All three regions' tests are evaluated and the region picks among the results: a warp holds
  // lanes of all three regions almost always, so branches would run all three blocks anyway.  Each
  // test compares the same doubles with the same relation as the published branches.
  {  // tetrahedron at (0,0,0)
    const bool b_z = xins >= yins && zins > yins, a_z = xins < yins && zins > xins;
    const double a_score = a_z ? zins : xins, b_score = b_z ? zins : yins;
    const int a_point = a_z ? 0x04 : 0x01, b_point = b_z ? 0x04 : 0x02;
    const double wins = 1 - in_sum;
    const int near = noise_bit((b_score > a_score) ? b_point : a_point);
    id = (wins > a_score || wins > b_score) ? near : 3 + noise_bit(7 ^ (a_point | b_point));
  }
  {  // tetrahedron at (1,1,1)
    const bool b_z = xins <= yins && zins < yins, a_z = xins > yins && zins < xins;
    const double a_score = a_z ? zins : xins, b_score = b_z ? zins : yins;
    const int a_point = a_z ? 0x03 : 0x06, b_point = b_z ? 0x03 : 0x05;
    const double wins = 3 - in_sum;
    const int near = 6 + noise_bit(7 ^ ((b_score < a_score) ? b_point : a_point));
    const int id_far = (wins < a_score || wins < b_score) ? near : 9 + noise_bit(a_point & b_point);
    id = in_sum <= 1 ? id : id_far;
  }
  {  // octahedron in between
    const double p1 = xins + yins, p2 = xins + zins, p3 = yins + zins;
    const bool a_far0 = p1 > 1, b_far0 = p2 > 1, far3 = p3 > 1;
    const double a_score = a_far0 ? p1 - 1 : 1 - p1, b_score = b_far0 ? p2 - 1 : 1 - p2;
    const double score = far3 ? p3 - 1 : 1 - p3;
    const bool to_a = a_score <= b_score && a_score < score, to_b = a_score > b_score && b_score < score;
    const int p3_point = far3 ? 0x06 : 0x01;
    const int a_point = to_a ? p3_point : (a_far0 ? 0x03 : 0x04);
    const int b_point = to_b ? p3_point : (b_far0 ? 0x05 : 0x02);
    const bool a_far = to_a ? far3 : a_far0, b_far = to_b ? far3 : b_far0;
    const int c1 = a_far ? a_point : b_point, c2 = a_far ? b_point : a_point;
    const int id_same = a_far ? 12 + noise_bit(a_point & b_point) : 15 + noise_bit(7 ^ (a_point | b_point));
    const int id_oct = a_far == b_far ? id_same : 18 + 3 * noise_bit(7 ^ c1) + noise_bit(c2);
    const bool oct = !(in_sum <= 1) && !(in_sum >= 2);
    id = oct ? id_oct : id;
    member = in_sum <= 1 ? 0x0Fu : in_sum >= 2 ? 0xF0u : 0x7Eu;
  }

  // the leaf as data: lattice offsets and displacements of the two extra vertices
  if (case_out) *case_out = id;  // tests only
  const uint64_t leaf = t.c->ext[id];
  const uint32_t leaf0 = (uint32_t)leaf, leaf1 = (uint32_t)(leaf >> 24);
#define CR_NOISE_EXT(W, AXIS, D0, SB, OUT_D, OUT_S)                                       \
  {                                                                                       \
    const int b_ = (int)(((W) >> (8 * (AXIS))) & 0xFFu);                                  \
    const int A1_ = b_ & 3, k_ = (b_ >> 2) & 3, C_ = b_ >> 4;  /* A1_ = A + 1 */          \
    OUT_D = (((D0) - t.c->small[A1_]) - t.c->ksq[k_]) - t.c->small[C_ + 1];               \
    OUT_S = (SB) + A1_ - 1 + C_;                                                          \
  }
  double dx_ext0, dy_ext0, dz_ext0, dx_ext1, dy_ext1, dz_ext1;
  int xsv_ext0, ysv_ext0, zsv_ext0, xsv_ext1, ysv_ext1, zsv_ext1;
  CR_NOISE_EXT(leaf0, 0, dx0, xsb, dx_ext0, xsv_ext0)
  CR_NOISE_EXT(leaf0, 1, dy0, ysb, dy_ext0, ysv_ext0)
  CR_NOISE_EXT(leaf0, 2, dz0, zsb, dz_ext0, zsv_ext0)
  CR_NOISE_EXT(leaf1, 0, dx0, xsb, dx_ext1, xsv_ext1)
  CR_NOISE_EXT(leaf1, 1, dy0, ysb, dy_ext1, ysv_ext1)
  CR_NOISE_EXT(leaf1, 2, dz0, zsb, dz_ext1, zsv_ext1)
#undef CR_NOISE_EXT

  // cube vertices in the common order; displacement (d0 - {0,1}) - m * SQ, m = i + j + k
  double value = 0;
  const double s1 = SQ, s2 = 2 * SQ, s3 = 3 * SQ;
  const double ax0 = dx0 - 0, ax1 = dx0 - 1, ay0 = dy0 - 0, ay1 = dy0 - 1, az0 = dz0 - 0, az1 = dz0 - 1;
  CR_NOISE_CONTRIB(member & 0x01u, xsb + 0, ysb + 0, zsb + 0, dx0, dy0, dz0)
  { const double dx = ax1 - s1, dy = ay0 - s1, dz = az0 - s1;
    CR_NOISE_CONTRIB(member & 0x02u, xsb + 1, ysb + 0, zsb + 0, dx, dy, dz) }
  { const double dx = ax0 - s1, dy = ay1 - s1, dz = az0 - s1;
    CR_NOISE_CONTRIB(member & 0x04u, xsb + 0, ysb + 1, zsb + 0, dx, dy, dz) }
  { const double dx = ax0 - s1, dy = ay0 - s1, dz = az1 - s1;
    CR_NOISE_CONTRIB(member & 0x08u, xsb + 0, ysb + 0, zsb + 1, dx, dy, dz) }
  { const double dx = ax1 - s2, dy = ay1 - s2, dz = az0 - s2;
    CR_NOISE_CONTRIB(member & 0x10u, xsb + 1, ysb + 1, zsb + 0, dx, dy, dz) }
  { const double dx = ax1 - s2, dy = ay0 - s2, dz = az1 - s2;
    CR_NOISE_CONTRIB(member & 0x20u, xsb + 1, ysb + 0, zsb + 1, dx, dy, dz) }
  { const double dx = ax0 - s2, dy = ay1 - s2, dz = az1 - s2;
    CR_NOISE_CONTRIB(member & 0x40u, xsb + 0, ysb + 1, zsb + 1, dx, dy, dz) }
  { const double dx = ax1 - s3, dy = ay1 - s3, dz = az1 - s3;
    CR_NOISE_CONTRIB(member & 0x80u, xsb + 1, ysb + 1, zsb + 1, dx, dy, dz) }
  CR_NOISE_CONTRIB(true, xsv_ext0, ysv_ext0, zsv_ext0, dx_ext0, dy_ext0, dz_ext0)
  CR_NOISE_CONTRIB(true, xsv_ext1, ysv_ext1, zsv_ext1, dx_ext1, dy_ext1, dz_ext1)
  return value / 103.0;
}

}  // namespace cr
