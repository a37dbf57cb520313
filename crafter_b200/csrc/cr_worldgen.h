// World generation: Env.reset (env.py:70-81) + worldgen.generate_world (worldgen.py:10-91).
//
// A world depends only on (env seed, episode), so the world of an env's NEXT episode is generated
// ahead of time into `next_*` buffers, off the critical path of the step, and `wg_install_*` swaps
// it in when the episode ends.
//   wg_seed      one warp per world: episode, world seed, simplex seed, permutation table
//   wg_material  one thread per cell: FP64 simplex terrain (pass 1, worldgen.py:21-61)
//   wg_object    one thread per cell: initial creature decision (pass 2, worldgen.py:64-76);
//                the calling kernel turns the per-cell decisions into slots with an ordered
//                prefix sum so that slot order == x-major cell order (worldgen.py:16-18)
//   wg_install_* copy the prefetched world into the live state + Player / Env reset
#pragma once
#include "cr_common.h"
#include "cr_noise.h"

namespace cr {

constexpr uint8_t TUNNEL_BIT = 0x80;  // `tunnels[x, y]` (worldgen.py:12) carried in mat bit 7
constexpr int OBJ_SHIFT = 4;          // bits 4-5 of a freshly generated cell: 0 none, 1 cow, 2 zombie, 3 skeleton
constexpr uint8_t MAT_MASK = 0x0F;

#ifdef CR_HOSTSIM
CR_DEV void cr_atomic_or(uint32_t *p, uint32_t v) { *p |= v; }
CR_DEV int cr_atomic_add_shared(int32_t *p, int v) { int o = *p; *p += v; return o; }
#else
CR_DEV void cr_atomic_or(uint32_t *p, uint32_t v) { atomicOr(p, v); }
CR_DEV int cr_atomic_add_shared(int32_t *p, int v) { return atomicAdd(p, v); }
#endif

struct SeedScratch {  // per-warp shared memory of the seeding kernel
  uint64_t lcg[256];
  uint16_t r[256];
  uint8_t source[256];
};

// env.py:72-74 + worldgen.py:11: world seed, simplex seed and permutation table of a world.
//   ahead = 0  the world about to be generated (episode = live episode + 1); a no-op when an
//              earlier ahead pass prepared it and wg_install_player promoted it (NM_SEEDED).
//   ahead = 1  the world after the one just generated; runs next to k_wg_obj, off the chain.
// One warp per world: lane 0 walks the 64-bit LCG, all lanes reduce the states to swap indices
// (64-bit modulo is the expensive part), lane 0 applies the serial shuffle in shared memory.
// worldgen.py:11 + the `opensimplex` constructor: simplex seed drawn from the world's keyed stream,
// 64-bit LCG, serial shuffle.  One warp: lane 0 walks the LCG, all lanes reduce the states to swap
// indices (64-bit modulo is the expensive part), lane 0 applies the serial shuffle in shared memory.
CR_DEV void wg_perm(uint32_t ws, uint8_t *perm, int lane, SeedScratch &S) {
  if (lane == 0) {
    Rng r = rng_ctx(ws, D_SEED, 0);
    uint64_t s = (uint64_t)rng_randint(r, 2147483647u);  // worldgen.py:11
    for (int k = 0; k < 3; ++k) s = s * 6364136223846793005ULL + 1442695040888963407ULL;
    for (int i = 255; i >= 0; --i) {
      s = s * 6364136223846793005ULL + 1442695040888963407ULL;
      S.lcg[i] = s;
    }
  }
  for (int i = lane; i < 256; i += CR_LANES) S.source[i] = (uint8_t)i;
#ifndef CR_HOSTSIM
  __syncwarp();
#endif
  for (int i = lane; i < 256; i += CR_LANES) {
    // Python: int((seed + 31) % (i + 1)) on an unbounded signed int, floored modulo.
    int64_t n = i + 1;
    int64_t a = (int64_t)S.lcg[i] % n;
    int64_t r = (a + 31 % n) % n;
    if (r < 0) r += n;
    S.r[i] = (uint16_t)r;
  }
#ifndef CR_HOSTSIM
  __syncwarp();
#endif
  if (lane == 0) {
    for (int i = 255; i >= 0; --i) {
      int r = S.r[i];
      perm[i] = S.source[r];
      S.source[r] = S.source[i];
    }
  }
}

CR_DEV uint8_t *wg_perm_of(const State &st, int env, int episode) {
  return st.perm + ((size_t)env * 2 + (episode & 1)) * 256;
}

CR_DEV void wg_seed(const Geom &g, const State &st, int env, int lane, SeedScratch &S, int ahead) {
  const int32_t *ps = st.pstate + (size_t)env * PS_COUNT;
  int32_t *nm = st.next_meta + (size_t)env * NM_COUNT;
  const bool seeded = !ahead && nm[NM_SEEDED];  // promoted by wg_install_player (uniform across the warp)
  const int episode = ahead ? nm[NM_EPISODE] + 1 : ps[PS_EPISODE] + 1;
  cr_syncwarp();  // every lane has read the row before lane 0 rewrites it below (found by tests/simt)
  if (seeded) return;
  // Two tables per env, by episode parity: the ahead pass writes the one k_wg_mat is NOT reading, so it
  // runs beside the terrain of the world before it instead of behind it.
  uint8_t *perm = wg_perm_of(st, env, episode);
  uint32_t ws = 0;
  if (lane == 0) {
    ws = world_seed_of(g.seed + g.env_offset + env, episode);
    nm[ahead ? NM_AHEAD_EPISODE : NM_EPISODE] = episode;
    nm[ahead ? NM_AHEAD_WORLD_SEED : NM_WORLD_SEED] = (int32_t)ws;
    if (!ahead) nm[NM_SEEDED] = 1;
  }
  wg_perm(ws, perm, lane, S);  // only lane 0 uses `ws`
  if (ahead && lane == 0) nm[NM_AHEAD_VALID] = 1;
}

// worldgen.py:64-76.  `matbyte` still carries TUNNEL_BIT.  Returns EntType or T_NONE.
CR_DEV int wg_object(const Geom &g, uint32_t world_seed, int x, int y, uint8_t matbyte) {
  const int px = g.W / 2, py = g.H / 2;
  const int m = matbyte & MAT_MASK;
  if (!((WALKABLE >> m) & 1u)) return T_NONE;
  Rng rng = rng_ctx(world_seed, D_WG_OBJ, (uint32_t)(x * g.H + y));
  int ddx = x - px, ddy = y - py;
  double dist = sqrt((double)(ddx * ddx + ddy * ddy));
  if (dist > 3 && m == M_GRASS && rng_uniform(rng) > 0.985) return T_COW;
  if (dist > 10 && rng_uniform(rng) > 0.993) return T_ZOMBIE;
  if (m == M_PATH && (matbyte & TUNNEL_BIT) && rng_uniform(rng) > 0.95) return T_SKELETON;
  return T_NONE;
}

// ---- terrain: worldgen.py:21-61, a tile of cells per CTA, octaves evaluated from a work list ----
// The reference evaluates up to 11 simplex octaves per cell, lazily, one after another; which ones
// depends on the cell.  Here a CTA owns WG_TILE cells and proceeds in at most four rounds; in each
// round every unfinished cell posts the octaves its current phase needs, the (cell, octave) items
// are processed densely by all threads through ONE noise3 call site, and a per-cell combine step
// applies the reference's branches (with its uniform draws, in its order) and picks the next phase.
// The start, water and mountain octaves are evaluated together, and so are the tunnel / ore octaves.  Otherwise a cell evaluates a SUBSET of
// the reference's lazy set: an octave whose threshold test is and-ed with a condition that is already
// known to fail (`simplex(..) > 0 and uniform() > 0.8`, `simplex(..) > 0.15 and mountain > 0.3`) cannot
// change the cell, and the keyed draws do not depend on the order they are looked at -- so the cheap
// side is looked at first (wg_enter_tree, wg_enter_tunnel) and the noise is skipped.
#ifndef CR_WG_TILE
#define CR_WG_TILE 256
#endif
constexpr int WG_TILE = CR_WG_TILE;
constexpr int WG_N_OCTAVES = 28;  // phase * 4 + slot
// WP_START posts five octaves at once (slots 0-3 water / mountain, slot 4 start: octave codes 0..4),
// so a cell goes through at most four rounds: START, CAVE, TUNNEL, LAVA.  Only cells within a few
// cells of the map centre (start > 0.5, ~3 % of a 64 x 64 map) have no use for the four water /
// mountain values; evaluating them costs less than a round of its own.
enum WgPhase : int8_t { WP_DONE = -1, WP_START = 0, WP_CAVE = 2, WP_SAND, WP_TREE, WP_TUNNEL, WP_LAVA };
constexpr int WG_ROUNDS = 4, WG_SLOTS = 5;

enum WgOctaveKind { WO_PLAIN = 0, WO_TUNNEL_H = 1, WO_TUNNEL_V = 2 };

// a / d for r = 1 / d: the product's error is removed with the exact remainder (Markstein).  This is
// the correctly rounded quotient -- the same double as `a / d` -- for every a a map side < 32768 makes
// (x or 2x over d in {3, 5, 6, 7, 8, 9, 15}, x / 5 over 3; all checked by tests/test_noise_boundaries.py),
// in three FP64 instructions where `/` takes a reciprocal, Newton steps and a range check.
CR_DEV double wg_div(double a, double d, double r) {
  const double q = a * r;
  return fma(fma(-q, d, a), r, q);
}

// An octave's arguments as data: per axis the numerator's factor and the divisor with its reciprocal;
// `again` = 1 / 2: the x / y quotient is divided by 3 once more (the tunnel octaves).
struct WgOctave {
  double dx, rx, dy, ry, z;
  int mx, my, again;
};

CR_DEV WgOctave wg_octave(uint32_t code) {
  const int size = code & 15, kind = code >> 8;
  WgOctave o;
  o.mx = kind == WO_TUNNEL_H ? 2 : 1;
  o.my = kind == WO_TUNNEL_V ? 2 : 1;
  o.dx = kind == WO_TUNNEL_V ? 5.0 : (double)size;
  o.dy = kind == WO_TUNNEL_H ? 5.0 : (double)size;
  o.rx = 1 / o.dx;
  o.ry = 1 / o.dy;
  o.z = (double)((code >> 4) & 15);
  o.again = kind == WO_TUNNEL_V ? 1 : kind == WO_TUNNEL_H ? 2 : 0;
  return o;
}

struct WgTile {  // shared memory of one CTA
  double start[WG_TILE], water[WG_TILE], mountain[WG_TILE];
  double v[WG_TILE][4];
  uint16_t items[WG_TILE * WG_SLOTS];  // cell * 8 + slot
  int32_t n_items;
  int8_t phase[WG_TILE];
  uint8_t need[WG_TILE];    // WP_TUNNEL: which of the four octaves can still change the cell (bit = slot)
  uint8_t result[WG_TILE];
  WgOctave oct[WG_N_OCTAVES];  // wg_octave(wg_octave_code(i))
};

// octaves (bit = slot) a cell in `phase` posts
CR_DEV unsigned wg_phase_slots(int phase, unsigned need) {
  return phase == WP_START ? 0x1Fu : phase == WP_TUNNEL ? need : 1u;
}

// worldgen.py:49-58 below the two tunnel tests, as a function of the two ore thresholds
// (`coal` = simplex(x, y, 1, 8) > 0, `iron` = simplex(x, y, 2, 6) > 0.4) and the cell's first three keyed
// draws: a material, or WG_ORE_LAVA = "ask the lava octave".  A draw is consumed only behind a true
// threshold, exactly like the reference's `and`.
constexpr int WG_ORE_LAVA = 0x40;
struct WgDraws { double u0, u1, u2; };
CR_DEV int wg_ore(bool coal, bool iron, double mountain, const WgDraws &u) {
  int k = 0;  // draws consumed so far
  if (coal) { if (u.u0 > 0.85) return M_COAL; k = 1; }
  if (iron) { if ((k ? u.u1 : u.u0) > 0.75) return M_IRON; ++k; }
  if (mountain > 0.18 && (k == 0 ? u.u0 : k == 1 ? u.u1 : u.u2) > 0.994) return M_DIAMOND;
  if (mountain > 0.3) return WG_ORE_LAVA;
  return M_STONE;
}
CR_DEV WgDraws wg_ore_draws(uint32_t world_seed, const Geom &g, int x, int y) {
  Rng rng = rng_ctx(world_seed, D_WG_MAT, (uint32_t)(x * g.H + y));
  WgDraws u;
  u.u0 = rng_uniform(rng); u.u1 = rng_uniform(rng); u.u2 = rng_uniform(rng);
  return u;
}
// -> WP_TUNNEL: both tunnel octaves, and each ore octave only if its threshold can change wg_ore's answer
CR_DEV int wg_enter_tunnel(const Geom &g, uint32_t world_seed, int x, int y, double mountain, WgTile &T, int c) {
  const WgDraws u = wg_ore_draws(world_seed, g, x, y);
  const int f00 = wg_ore(false, false, mountain, u), f01 = wg_ore(false, true, mountain, u);
  const int f10 = wg_ore(true, false, mountain, u), f11 = wg_ore(true, true, mountain, u);
  unsigned need = 3u;
  if (f00 != f10 || f01 != f11) need |= 4u;  // coal
  if (f00 != f01 || f10 != f11) need |= 8u;  // iron
  T.need[c] = (uint8_t)need;
  return WP_TUNNEL;
}
// -> WP_TREE only if the draw lets a tree grow at all (worldgen.py:60); else the cell is grass
CR_DEV int wg_enter_tree(const Geom &g, uint32_t world_seed, int x, int y) {
  Rng rng = rng_ctx(world_seed, D_WG_MAT, (uint32_t)(x * g.H + y));
  return rng_uniform(rng) > 0.8 ? WP_TREE : WP_DONE;  // WP_DONE: result stays M_GRASS
}

// _simplex(x, y, z, size) -> noise3(x / size, y / size, z) for the octave (phase, slot) asks for
// (worldgen.py:27-60,79-91).  The items of a warp ask for different octaves, so the octave is data
// (wg_octave_code -> wg_octave, staged once per CTA as T.oct[]) and every lane runs the same
// divisions: one per axis, and a third that only the tunnel octaves `(2x, y/5, 7, 3)` /
// `(x/5, 2y, 7, 3)` keep.
// size | z << 4 | kind << 8
CR_DEV uint16_t wg_octave_code(int code) {
  int size = 5, z = 6, kind = WO_PLAIN;                               // lava     (x, y, 6, 5)
  switch (code) {
    case WP_START * 4 + 0: size = 15; z = 3; break;                   // water    (x, y, 3, 15)
    case WP_START * 4 + 1: size = 5; z = 3; break;                    // water    (x, y, 3, 5)
    case WP_START * 4 + 2: size = 15; z = 0; break;                   // mountain (x, y, 0, 15)
    case WP_START * 4 + 3: size = 5; z = 0; break;                    // mountain (x, y, 0, 5)
    case WP_START * 4 + 4: size = 3; z = 8; break;                    // start    (x, y, 8, 3)
    case WP_CAVE * 4: size = 7; z = 6; break;                         // cave     (x, y, 6, 7)
    case WP_SAND * 4: size = 9; z = 4; break;                         // sand     (x, y, 4, 9)
    case WP_TREE * 4: size = 7; z = 5; break;                         // tree     (x, y, 5, 7)
    case WP_TUNNEL * 4 + 0: size = 3; z = 7; kind = WO_TUNNEL_H; break;  // (2x, y/5, 7, 3)
    case WP_TUNNEL * 4 + 1: size = 3; z = 7; kind = WO_TUNNEL_V; break;  // (x/5, 2y, 7, 3)
    case WP_TUNNEL * 4 + 2: size = 8; z = 1; break;                   // coal     (x, y, 1, 8)
    case WP_TUNNEL * 4 + 3: size = 6; z = 2; break;                   // iron     (x, y, 2, 6)
    default: break;
  }
  return (uint16_t)(size | (z << 4) | (kind << 8));
}

CR_DEV void wg_octave_args(const WgOctave &o, int x, int y, double &ax, double &ay, double &az) {
  const double qx = wg_div((double)(o.mx * x), o.dx, o.rx), qy = wg_div((double)(o.my * y), o.dy, o.ry);
  const double q3 = wg_div(o.again == 1 ? qx : qy, 3.0, 1.0 / 3.0);
  ax = o.again == 1 ? q3 : qx;
  ay = o.again == 2 ? q3 : qy;
  az = o.z;
}

// worldgen.py:27-48 once `start` and the water / mountain octaves (v[0..3]) are known: the next phase.
CR_DEV int wg_water_mountain(const Geom &g, uint32_t world_seed, int x, int y, WgTile &T, int c, double start,
                             int &result) {
  const double *v = T.v[c];
  double water = (0 + 1 * v[0]) + 0.15 * v[1];  // {15: 1, 5: 0.15}, unnormalised
  water = water + 0.1;
  water -= 2 * start;
  double mountain = (0 + 1 * v[2]) + 0.3 * v[3];  // {15: 1, 5: 0.3}
  mountain /= (1 + 0.3);
  mountain -= 4 * start + 0.3 * water;
  T.water[c] = water; T.mountain[c] = mountain;
  if (mountain > 0.15)  // caves need `simplex(x, y, 6, 7) > 0.15 and mountain > 0.3` (worldgen.py:40)
    return mountain > 0.3 ? WP_CAVE : wg_enter_tunnel(g, world_seed, x, y, mountain, T, c);
  if (0.25 < water && water <= 0.35) return WP_SAND;
  if (0.3 < water) { result = M_WATER; return WP_DONE; }
  return wg_enter_tree(g, world_seed, x, y);
}

// The reference's branch structure for one cell once the octaves of its phase are in v[].
CR_DEV void wg_combine(const Geom &g, uint32_t world_seed, int x, int y, WgTile &T, int c) {
  const double *v = T.v[c];
  int phase = T.phase[c], result = M_GRASS;
  switch (phase) {
    case WP_START: {
      int ddx = x - g.W / 2, ddy = y - g.H / 2;  // player at the centre, env.py:71
      double start = 4 - sqrt((double)(ddx * ddx + ddy * ddy));
      start += 2 * T.start[c];  // the start octave (slot 4)
      start = 1 / (1 + exp(-start));
      T.start[c] = start;
      phase = start > 0.5 ? WP_DONE : wg_water_mountain(g, world_seed, x, y, T, c, start, result);  // DONE: grass
    } break;
    case WP_CAVE:  // mountain > 0.3 here
      if (v[0] > 0.15) { result = M_PATH; phase = WP_DONE; }
      else phase = wg_enter_tunnel(g, world_seed, x, y, T.mountain[c], T, c);
      break;
    case WP_SAND:
      if (v[0] > -0.2) { result = M_SAND; phase = WP_DONE; }
      else if (0.3 < T.water[c]) { result = M_WATER; phase = WP_DONE; }
      else phase = wg_enter_tree(g, world_seed, x, y);
      break;
    case WP_TREE:  // the draw said > 0.8 (wg_enter_tree)
      result = v[0] > 0 ? M_TREE : M_GRASS;
      phase = WP_DONE;
      break;
    case WP_TUNNEL: {
      const double mountain = T.mountain[c];
      const unsigned need = T.need[c];
      phase = WP_DONE;
      if (v[0] > 0.4) result = M_PATH | TUNNEL_BIT;        // horizontal tunnel
      else if (v[1] > 0.4) result = M_PATH | TUNNEL_BIT;   // vertical tunnel
      else {
        const WgDraws u = wg_ore_draws(world_seed, g, x, y);
        // an octave that was not asked for cannot change the answer: any value does
        const int r = wg_ore((need & 4u) && v[2] > 0, (need & 8u) && v[3] > 0.4, mountain, u);
        if (r == WG_ORE_LAVA) phase = WP_LAVA;
        else result = r;
      }
    } break;
    default:  // WP_LAVA
      result = v[0] > 0.35 ? M_LAVA : M_STONE;
      phase = WP_DONE;
      break;
  }
  T.phase[c] = (int8_t)phase;
  if (phase == WP_DONE) T.result[c] = (uint8_t)result;
}

// Terrain of cells [cell0, cell0 + ncell) of one world into `out` (TUNNEL_BIT kept in bit 7).
// Called by all `nthreads` threads of the CTA (block-generic; the host-sim runs it with one).
CR_DEV void wg_material_tile(const Geom &g, const NoiseTables &t, uint32_t world_seed, uint8_t *out,
                             int cell0, int ncell, int tid, int nthreads, WgTile &T) {
  for (int c = tid; c < ncell; c += nthreads) T.phase[c] = WP_START;
  for (int i = tid; i < WG_N_OCTAVES; i += nthreads) T.oct[i] = wg_octave(wg_octave_code(i));
  cr_syncblock();
  for (int round = 0; round < WG_ROUNDS; ++round) {
    if (tid == 0) T.n_items = 0;
    cr_syncblock();
    for (int c = tid; c < ncell; c += nthreads) {
      const int phase = T.phase[c];
      if (phase == WP_DONE) continue;
      const unsigned slots = wg_phase_slots(phase, T.need[c]);
      int at = cr_atomic_add_shared(&T.n_items, cr_popc(slots));
      for (int s2 = 0; s2 < WG_SLOTS; ++s2)
        if ((slots >> s2) & 1u) T.items[at++] = (uint16_t)(c * 8 + s2);
    }
    cr_syncblock();
    const int n = T.n_items;
    if (n == 0) break;  // uniform
    for (int it = tid; it < n; it += nthreads) {
      const int c = T.items[it] >> 3, slot = T.items[it] & 7;
      const int cell = cell0 + c, x = cell / g.H, y = cell - x * g.H;
      double ax, ay, az;
      wg_octave_args(T.oct[T.phase[c] * 4 + slot], x, y, ax, ay, az);
      const double value = noise3(t, ax, ay, az);
      if (slot < 4) T.v[c][slot] = value;
      else T.start[c] = value;
    }
    cr_syncblock();
    for (int c = tid; c < ncell; c += nthreads) {
      if (T.phase[c] == WP_DONE) continue;
      const int cell = cell0 + c, x = cell / g.H, y = cell - x * g.H;
      wg_combine(g, world_seed, x, y, T, c);
    }
    cr_syncblock();
  }
  // Pass 2 of worldgen (initial creatures, worldgen.py:64-76) only looks at the cell itself, so its
  // decision rides along in the byte: bits 0-3 material, 4-5 creature (OBJ_SHIFT), 7 tunnel.  The
  // slot order of the creatures is fixed later by an ordered prefix sum (k_wg_obj).
  for (int c = tid; c < ncell; c += nthreads) {
    const int cell = cell0 + c, x = cell / g.H, y = cell - x * g.H;
    const uint8_t m = T.result[c];
    const int type = wg_object(g, world_seed, x, y, m);
    out[cell] = (uint8_t)(m | ((type ? type - 1 : 0) << OBJ_SHIFT));
  }
}

CR_DEV Ent wg_make_entity(int type, int x, int y) {  // objects.py:266-268,284-288,317-321
  Ent e;
  e.type = (uint8_t)type;
  e.health = (int8_t)(type == T_ZOMBIE ? 5 : 3);
  e.x = (int16_t)x; e.y = (int16_t)y; e.aux = 0;
  return e;
}

// ---- install: prefetched world -> live state (World.reset engine.py:33-39 + env.py:70-81) -----
// Phase A (all threads): terrain copy, empty object map, empty touched set.
CR_DEV void wg_install_clear(const Geom &g, const State &st, int env, int tid, int nthreads) {
  uint8_t *mat = st.mat + (size_t)env * g.NC;
  const uint8_t *src = next_mat_of(st, g, env);
  uint16_t *objmap = st.objmap + (size_t)env * g.NC;
  uint32_t *touched = st.touched + (size_t)env * g.TW;
  if ((g.NC & 15) == 0) {  // rows of every env stay 16-byte aligned
    const uint64_t *s8 = reinterpret_cast<const uint64_t *>(src);
    uint64_t *d8 = reinterpret_cast<uint64_t *>(mat), *o8 = reinterpret_cast<uint64_t *>(objmap);
    for (int i = tid; i < g.NC / 8; i += nthreads) d8[i] = s8[i];
    for (int i = tid; i < g.NC / 4; i += nthreads) o8[i] = 0;
  } else {
    for (int c = tid; c < g.NC; c += nthreads) { mat[c] = src[c]; objmap[c] = 0; }
  }
  for (int c = tid; c < g.TW; c += nthreads) touched[c] = 0;
}

// Phase A for the map rows x0 <= x < x1 only (k_install splits an env over its chunk columns).
CR_DEV void wg_install_clear_rows(const Geom &g, const State &st, int env, int x0, int x1, int tid, int nthreads) {
  const int c0 = x0 * g.H, n = (x1 - x0) * g.H;
  uint8_t *mat = st.mat + (size_t)env * g.NC + c0;
  const uint8_t *src = next_mat_of(st, g, env) + c0;
  uint16_t *objmap = st.objmap + (size_t)env * g.NC + c0;
  if (((g.NC | c0 | n) & 15) == 0) {  // rows of every env and of every column stay 16-byte aligned
    const uint64_t *s8 = reinterpret_cast<const uint64_t *>(src);
    uint64_t *d8 = reinterpret_cast<uint64_t *>(mat), *o8 = reinterpret_cast<uint64_t *>(objmap);
    for (int i = tid; i < n / 8; i += nthreads) d8[i] = s8[i];
    for (int i = tid; i < n / 4; i += nthreads) o8[i] = 0;
  } else {
    for (int c = tid; c < n; c += nthreads) { mat[c] = src[c]; objmap[c] = 0; }
  }
}

// Phase B (all threads, after a barrier): creatures into slots 2.., object map, touched chunks.
CR_DEV void wg_install_scatter(const Geom &g, const State &st, int env, int tid, int nthreads) {
  const int n = next_meta_of(st, env)[NM_NSLOTS];
  const Ent *src = next_ents_of(st, g, env);
  Ent *ents = st.ents + (size_t)env * g.CAP;
  uint16_t *objmap = st.objmap + (size_t)env * g.NC;
  uint32_t *touched = st.touched + (size_t)env * g.TW;
  for (int s = 2 + tid; s < n; s += nthreads) {
    Ent e = src[s];
    ents[s] = e;
    objmap[e.x * g.H + e.y] = (uint16_t)s;
    int ch = (e.x / CHUNK) * g.ncy + (e.y / CHUNK);
    cr_atomic_or(&touched[ch >> 5], 1u << (ch & 31));
  }
}

// Phase C (one thread): Player + per-episode scalars, env.py:75-79, objects.py:70-82,
// data.yaml:39-55; consumes the prefetched world.
// Player + per-episode scalars of a fresh episode, env.py:75-79, objects.py:70-82, data.yaml:39-55.
CR_DEV void wg_fresh_player(const Geom &g, const State &st, int env, int n_slots, int episode,
                            int world_seed) {
  int32_t *ps = st.pstate + (size_t)env * PS_COUNT;
  int32_t *inv = st.inventory + (size_t)env * N_ITEMS;
  int32_t *ach = st.achievements + (size_t)env * N_ACH;
  for (int i = 0; i < N_ITEMS; ++i) inv[i] = i < 4 ? 9 : 0;
  for (int i = 0; i < N_ACH; ++i) ach[i] = 0;
  ps[PS_HUNGER2] = 0; ps[PS_THIRST2] = 0; ps[PS_FATIGUE] = 0; ps[PS_RECOVER2] = 0;
  ps[PS_SLEEPING] = 0; ps[PS_P_LAST_HEALTH] = 9; ps[PS_LAST_HEALTH] = 9; ps[PS_UNLOCKED] = 0;
  ps[PS_NSLOTS] = n_slots; ps[PS_STEP] = 0;
  ps[PS_EPISODE] = episode; ps[PS_WORLD_SEED] = world_seed;
  ps[PS_PX] = g.W / 2; ps[PS_PY] = g.H / 2;
  st.ep_return[(size_t)env * 2] = 0.0;
  Ent p;
  p.type = T_PLAYER; p.health = 9; p.x = (int16_t)(g.W / 2); p.y = (int16_t)(g.H / 2);
  p.aux = 3;  // facing (0, 1) = down, objects.py:72
  Ent *ents = st.ents + (size_t)env * g.CAP;
  ents[1] = p;
  ents[0].type = T_NONE;
  st.objmap[(size_t)env * g.NC + (g.W / 2) * g.H + g.H / 2] = 1;  // env.py:76-78
  int ch = ((g.W / 2) / CHUNK) * g.ncy + ((g.H / 2) / CHUNK);
  cr_atomic_or(&st.touched[(size_t)env * g.TW + (ch >> 5)], 1u << (ch & 31));
}

// Phase C (one thread): consumes the prefetched world.
CR_DEV void wg_install_player(const Geom &g, const State &st, int env) {
  int32_t *nm = st.next_meta + (size_t)env * NM_COUNT;
  wg_fresh_player(g, st, env, nm[NM_NSLOTS], nm[NM_EPISODE], nm[NM_WORLD_SEED]);
  if (nm[NM_VALID] & 2) st.pstate[(size_t)env * PS_COUNT + PS_ERROR] |= ERR_SLOT_OVERFLOW;  // found by k_wg_obj
  nm[NM_VALID] = 0;
  // the seed prepared ahead (next to k_wg_obj) becomes the seed of the world to generate next
  nm[NM_SEEDED] = nm[NM_AHEAD_VALID];
  if (nm[NM_AHEAD_VALID]) {
    nm[NM_EPISODE] = nm[NM_AHEAD_EPISODE];
    nm[NM_WORLD_SEED] = nm[NM_AHEAD_WORLD_SEED];
    nm[NM_AHEAD_VALID] = 0;
  }
}

}  // namespace cr
