"""TEST INFRASTRUCTURE shared by the fixture generator (tools/make_scenarios.py) and the fixture replays
(tests/test_scenarios_golden.py: host-sim on CPU, the CUDA library on the GPU box;
tests/test_scenarios_vs_reference.py: the perturbation fuzz on the host-sim).

A *scenario* is a state that random rollouts rarely reach, built INSIDE a live reference env through
the reference's own World / object API (engine.py, objects.py), exported as a canonical state
(oracle/canon.py), loaded into an implementation and stepped with a fixed action list."""
import numpy as np

from crafter_b200 import state as state_lib

DIRS = ((-1, 0), (1, 0), (0, -1), (0, 1))  # objects.py:33-34
NOOP, LEFT, RIGHT, UP, DOWN, DO, SLEEP = range(7)
PLACE_STONE, PLACE_TABLE, PLACE_FURNACE, PLACE_PLANT = 7, 8, 9, 10
MAKE_WOOD_PICKAXE, MAKE_STONE_PICKAXE, MAKE_IRON_PICKAXE = 11, 12, 13
MAKE_WOOD_SWORD, MAKE_STONE_SWORD, MAKE_IRON_SWORD = 14, 15, 16
WALKABLE = ('grass', 'sand', 'path')


# ---- canonical state -> raw SoA arrays (layout: csrc/cr_common.h) --------------------------------
def raw_arrays(st, extras, area, capacity):
  """One env's canonical state `st` (+ extras: step, episode, world_seed) as the arrays of the SoA
  layout: mat u8[NC], objmap u16[NC], ents i64[CAP], inventory i32[16], achievements i32[22],
  pstate i32[16], touched u32[TW]."""
  W, H = area
  nch = -(-W // 12) * -(-H // 12)
  mat = np.ascontiguousarray(st['mat'], np.uint8).reshape(-1).copy()
  objmap = np.zeros(W * H, np.uint16)
  ents64 = np.zeros(capacity, np.int64)
  ents = ents64.view(state_lib.ENT_DTYPE)
  assert len(st['objs']) + 1 < capacity
  for k, (t, x, y, health, a, b) in enumerate(st['objs']):
    slot = k + 1
    ents[slot] = (t, min(health, 127), x, y, a)
    objmap[x * H + y] = slot
  p = st['player']
  ps = np.zeros(len(state_lib.PS), np.int32)
  PS = state_lib.PS
  ps[PS['hunger2']], ps[PS['thirst2']] = p[38], p[39]
  ps[PS['fatigue']], ps[PS['recover2']] = p[40], p[41]
  ps[PS['sleeping']] = p[42]
  ps[PS['player_last_health']] = p[44]
  ps[PS['player_x']], ps[PS['player_y']] = p[45], p[46]
  ps[PS['env_last_health']] = p[47]
  ps[PS['unlocked']] = np.int64(p[48]).astype(np.int32)
  ps[PS['n_slots']] = len(st['objs']) + 1
  ps[PS['step']] = extras['step']
  ps[PS['episode']] = extras['episode']
  ps[PS['world_seed']] = extras['world_seed']
  touched = np.zeros((nch + 31) // 32, np.uint32)
  for c in st['touched']:
    touched[c >> 5] |= np.uint32(1 << (c & 31))
  return dict(mat=mat, objmap=objmap, ents=ents64, inventory=np.asarray(p[:16], np.int32),
              achievements=np.asarray(p[16:38], np.int32), pstate=ps, touched=touched)


def load_numpy(state, i, raw):
  """Write `raw` into env i of a dict of numpy state arrays (tests/hostsim_env.HostSimEnv.state)."""
  for k, v in raw.items():
    state[k][i] = v


def load_torch(state, i, raw):
  """Write `raw` into env i of crafter_b200.Env.state (torch.cuda tensors)."""
  import torch
  signed = dict(objmap=np.int16, touched=np.int32)
  for k, v in raw.items():
    v = v.view(signed[k]) if k in signed else v
    state[k][i].copy_(torch.from_numpy(np.ascontiguousarray(v)))


# ---- packed fixture layout -----------------------------------------------------------------------
def pack(blob):
  """A fixture's s{i}_{key} members as one member per key: p_{key} (the arrays of every scenario,
  flattened and concatenated) and p_{key}_shapes (K, ndim).  Far fewer .npz members, and they
  compress better than one small member per scenario and key."""
  out, parts = {}, {}
  for k, v in blob.items():
    if k.startswith('meta_'):
      out[k] = v
    else:
      i, key = k[1:].split('_', 1)
      parts.setdefault(key, {})[int(i)] = np.asarray(v)
  for key, by_index in parts.items():
    arrays = [by_index[i] for i in range(len(by_index))]
    out[f'p_{key}'] = np.concatenate([a.reshape(-1) for a in arrays])
    out[f'p_{key}_shapes'] = np.array([a.shape for a in arrays], np.int64).reshape(len(arrays), arrays[0].ndim)
  return out


def unpack(z):
  """Inverse of pack: a dict with the s{i}_{key} members of the unpacked layout."""
  out = {k: z[k] for k in z.files if k.startswith('meta_')}
  for k in z.files:
    if k.startswith('p_') and not k.endswith('_shapes'):
      flat, at = z[k], 0
      for i, shape in enumerate(z[k + '_shapes']):
        n = int(np.prod(shape))
        out[f's{i}_{k[2:]}'] = flat[at:at + n].reshape(shape)
        at += n
  return out


# ---- helpers over the reference's API -------------------------------------------------------------
def flatten(env, x0, y0, x1, y1, material='grass'):
  """Rect [x0, x1) x [y0, y1) becomes `material`; every object but the player leaves it."""
  world, player = env._world, env._player
  W, H = world.area
  for x in range(max(0, x0), min(W, x1)):
    for y in range(max(0, y0), min(H, y1)):
      world[x, y] = material
      obj = world[(x, y)][1]
      if obj is not None and obj is not player:
        world.remove(obj)


def teleport(env, x, y, facing=(0, 1)):
  world, player = env._world, env._player
  obj = world[(x, y)][1]
  if obj is not None and obj is not player:
    world.remove(obj)
  if world[(x, y)][0] not in WALKABLE:
    world[x, y] = 'grass'
  if tuple(player.pos) != (x, y):
    world.move(player, (x, y))
  player.facing = facing


def give(env, **items):
  for k, v in items.items():
    env._player.inventory[k] = int(v)
  env._player._last_health = env._player.health
  env._last_health = env._player.health


def set_step(env, step):
  env._step = int(step)
  env._update_time()


def spawn(env, mods, kind, x, y, **attrs):
  objects, world = mods['objects'], env._world
  old = world[(x, y)][1]
  assert old is not env._player, 'scenario bug: spawning onto the player'
  if old is not None:
    world.remove(old)
  if kind in ('Zombie', 'Skeleton'):
    o = getattr(objects, kind)(world, (x, y), env._player)
  elif kind == 'Arrow':
    o = objects.Arrow(world, (x, y), attrs.pop('facing'))
  else:
    o = getattr(objects, kind)(world, (x, y))
  for k, v in attrs.items():
    setattr(o, k, v)
  world.add(o)
  return o


# ---- random perturbation (the fuzz) ---------------------------------------------------------------
def perturb(env, rs, mods):
  """Random edits of a reference env through World / object APIs (engine.py, objects.py)."""
  objects, world, player = mods['objects'], env._world, env._player
  W, H = world.area
  # terrain patches, including the materials that random walks seldom meet
  for _ in range(rs.randint(5, 40)):
    x, y = rs.randint(0, W), rs.randint(0, H)
    world[x, y] = rs.choice(['lava', 'water', 'table', 'furnace', 'tree', 'stone', 'coal', 'iron',
                             'diamond', 'grass', 'sand', 'path'])
  # teleport the player, often to an edge or corner
  for _ in range(20):
    x = rs.choice([0, 1, W - 2, W - 1, rs.randint(0, W)])
    y = rs.choice([0, 1, H - 2, H - 1, rs.randint(0, H)])
    if world[(x, y)][1] is None and world[(x, y)][0] in ('grass', 'sand', 'path'):
      world.move(player, (x, y))
      break
  px, py = player.pos
  for dx, dy in ((1, 0), (-1, 0), (0, 1), (0, -1), (1, 1)):  # useful neighbours
    x, y = px + dx, py + dy
    if 0 <= x < W and 0 <= y < H and world[(x, y)][1] is None and rs.rand() < 0.6:
      world[x, y] = rs.choice(['table', 'furnace', 'lava', 'water', 'tree', 'stone', 'iron', 'diamond', 'grass'])
  player.facing = [(-1, 0), (1, 0), (0, -1), (0, 1)][rs.randint(4)]
  # creatures around the player with odd attributes (dying mobs, loaded skeletons, ripe plants ...)
  for _ in range(rs.randint(3, 14)):
    x, y = px + rs.randint(-6, 7), py + rs.randint(-6, 7)
    if not (0 <= x < W and 0 <= y < H) or world[(x, y)][1] is not None:
      continue
    kind = rs.randint(5)
    mat = world[(x, y)][0]
    if kind == 0 and mat in ('grass', 'sand', 'path'):
      o = objects.Zombie(world, (x, y), player); o.health = rs.randint(0, 6); o.cooldown = rs.randint(0, 6)
    elif kind == 1 and mat in ('grass', 'sand', 'path'):
      o = objects.Skeleton(world, (x, y), player); o.health = rs.randint(0, 4); o.reload = rs.randint(0, 5)
    elif kind == 2 and mat in ('grass', 'sand', 'path'):
      o = objects.Cow(world, (x, y)); o.health = rs.randint(0, 4)
    elif kind == 3 and mat in ('grass', 'sand', 'path', 'water', 'lava'):
      o = objects.Arrow(world, (x, y), [(-1, 0), (1, 0), (0, -1), (0, 1)][rs.randint(4)])
    elif kind == 4 and mat == 'grass':
      o = objects.Plant(world, (x, y)); o.grown = rs.choice([0, 299, 300, 301, 500]); o.health = rs.randint(0, 2)
    else:
      continue
    world.add(o)
  for name in player.inventory:
    player.inventory[name] = int(rs.choice([0, 0, 1, 2, 5, 9]))
  player.inventory['health'] = int(rs.randint(1, 10))
  player.sleeping = bool(rs.rand() < 0.1)
  if rs.rand() < 0.5:
    player.inventory['energy'] = 9
  player._hunger, player._thirst = float(rs.randint(0, 26)), float(rs.randint(0, 21))
  player._fatigue, player._recover = int(rs.randint(-10, 31)), float(rs.randint(-15, 26))
  player._last_health = player.health
  env._last_health = player.health
  env._step = int(rs.choice([env._step, 140, 147, 200, 271, 299, 9]))
  env._update_time()


def fuzz_actions(rs, steps):
  return [int(rs.randint(0, 17)) if rs.rand() < 0.5 else
          int(rs.choice([5, 5, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16])) for _ in range(steps)]


# ---- directed scenarios: one per rule corner (SURVEY.md 8a quirks Q1-Q15) -------------------------
# Each builder edits a freshly reset reference env and returns the action list.
def d_craft_chain(env, mods, rs):
  """All six make_* next to table + furnace, then every pickaxe-gated collect, then place stone /
  table / furnace (objects.py:213-261, data.yaml:57-78)."""
  flatten(env, 6, 6, 15, 15)
  teleport(env, 10, 10, (0, 1))
  w = env._world
  w[9, 9] = 'table'; w[11, 11] = 'furnace'
  w[10, 11] = 'diamond'; w[11, 10] = 'iron'; w[9, 10] = 'coal'; w[10, 9] = 'stone'
  give(env, wood=9, stone=6, coal=3, iron=3)
  return [MAKE_WOOD_PICKAXE, MAKE_STONE_PICKAXE, MAKE_IRON_PICKAXE, MAKE_WOOD_SWORD, MAKE_STONE_SWORD,
          MAKE_IRON_SWORD, MAKE_IRON_SWORD, DO, RIGHT, DO, LEFT, DO, UP, DO, PLACE_STONE, DO, PLACE_TABLE,
          LEFT, PLACE_FURNACE, PLACE_STONE, PLACE_STONE, PLACE_STONE, PLACE_STONE, PLACE_FURNACE,
          DOWN, DOWN, PLACE_TABLE, PLACE_TABLE, MAKE_IRON_PICKAXE, NOOP]


def d_gated_collects_fail(env, mods, rs):
  """`do` on stone / coal / iron / diamond without the required pickaxe (objects.py:219-224)."""
  flatten(env, 6, 6, 15, 15)
  teleport(env, 10, 10, (0, 1))
  w = env._world
  w[10, 11] = 'diamond'; w[11, 10] = 'iron'; w[9, 10] = 'coal'; w[10, 9] = 'stone'
  give(env, wood_pickaxe=0, stone_pickaxe=0, iron_pickaxe=0, wood=0)
  return [DO, RIGHT, DO, LEFT, DO, UP, DO] + [MAKE_WOOD_PICKAXE, PLACE_TABLE, PLACE_STONE, PLACE_FURNACE, PLACE_PLANT, NOOP]


def _edge(x, y, facing):
  def build(env, mods, rs):
    W, H = env._world.area
    px, py = (x if x >= 0 else W + x), (y if y >= 0 else H + y)
    flatten(env, px - 3, py - 3, px + 4, py + 4)
    teleport(env, px, py, facing)
    w = env._world
    for dx, dy, m in ((1, 1, 'table'), (-1, -1, 'table'), (1, -1, 'furnace'), (-1, 1, 'furnace')):
      tx, ty = px + dx, py + dy
      if 0 <= tx < W and 0 <= ty < H:
        w[tx, ty] = m
    give(env, wood=9, stone=9, coal=9, iron=9, sapling=5)
    # crafting at the low edges is impossible (Q7, engine.py:95-103); placing / moving / hitting
    # towards the outside of the map is rejected (Q14)
    return [MAKE_WOOD_PICKAXE, MAKE_IRON_SWORD, PLACE_STONE, PLACE_TABLE, PLACE_PLANT, DO, LEFT, PLACE_STONE,
            DO, UP, PLACE_TABLE, DO, RIGHT, PLACE_FURNACE, DO, DOWN, PLACE_PLANT, DO, MAKE_STONE_PICKAXE,
            LEFT, LEFT, UP, UP, MAKE_WOOD_SWORD, RIGHT, RIGHT, DOWN, DOWN, MAKE_STONE_SWORD]
  return build


def d_lava_walk(env, mods, rs):
  """Walking into lava kills (Q8, objects.py:175-179): done with reward -0.9."""
  flatten(env, 6, 6, 15, 15)
  teleport(env, 10, 10, (0, 1))
  env._world[12, 10] = 'lava'
  return [RIGHT, NOOP, RIGHT, NOOP, NOOP]


def d_plants(env, mods, rs):
  """Saplings: place_plant, eating ripe / hitting unripe plants, plants eaten by neighbours
  (objects.py:190-194,405-411)."""
  flatten(env, 4, 4, 17, 17)
  teleport(env, 10, 10, (0, 1))
  give(env, sapling=3, food=3)
  spawn(env, mods, 'Plant', 11, 10, grown=301)
  spawn(env, mods, 'Plant', 9, 10, grown=299)
  spawn(env, mods, 'Plant', 10, 9, grown=300)
  spawn(env, mods, 'Plant', 14, 14, grown=5)
  spawn(env, mods, 'Cow', 14, 15)
  spawn(env, mods, 'Plant', 6, 6, grown=5, health=3)
  spawn(env, mods, 'Zombie', 6, 7, cooldown=3)
  return [PLACE_PLANT, DO, RIGHT, DO, DO, LEFT, DO, DO, DO, UP, DO, DO, DO, DOWN, DO, PLACE_PLANT,
          NOOP, NOOP, NOOP, RIGHT, DO]


def d_sapling_luck(env, mods, rs):
  """`do` on grass draws one uniform per try, sapling with p = 0.1 (data.yaml:64, objects.py:226)."""
  flatten(env, 6, 6, 15, 15)
  teleport(env, 10, 10, (0, 1))
  return [DO] * 45 + [PLACE_PLANT, DOWN, PLACE_PLANT]


def d_water_lava_stone(env, mods, rs):
  """Drinking resets thirst before the collect table (Q6); stone can be placed on water and lava."""
  flatten(env, 6, 6, 15, 15)
  teleport(env, 10, 10, (1, 0))
  w = env._world
  w[10, 11] = 'water'; w[11, 10] = 'lava'; w[9, 10] = 'water'
  give(env, drink=2, stone=3, wood_pickaxe=1)
  env._player._thirst = 19.0
  return [PLACE_STONE, DO, DOWN, DO, DO, DO, PLACE_STONE, DO, LEFT, PLACE_TABLE, PLACE_STONE, LEFT, DO, LEFT]


def d_arrows(env, mods, rs):
  """Arrows against everything (objects.py:373-384): table / furnace turn to path, any object
  loses 2 health (player, plant, cow, another arrow), water / lava are flown over, map edge."""
  flatten(env, 0, 0, 30, 30)
  teleport(env, 10, 10, (0, 1))
  w = env._world
  w[20, 5] = 'table'; spawn(env, mods, 'Arrow', 17, 5, facing=(1, 0))
  w[20, 7] = 'furnace'; spawn(env, mods, 'Arrow', 18, 7, facing=(1, 0))
  w[20, 9] = 'stone'; spawn(env, mods, 'Arrow', 18, 9, facing=(1, 0))
  w[19, 11] = 'water'; w[20, 11] = 'lava'; spawn(env, mods, 'Arrow', 17, 11, facing=(1, 0))
  spawn(env, mods, 'Arrow', 2, 13, facing=(-1, 0))   # leaves the map on the left
  spawn(env, mods, 'Arrow', 13, 1, facing=(0, -1))   # leaves the map at the top
  spawn(env, mods, 'Arrow', 7, 10, facing=(1, 0))    # hits the player
  spawn(env, mods, 'Arrow', 10, 14, facing=(0, -1))  # hits the player from below
  spawn(env, mods, 'Plant', 15, 15); spawn(env, mods, 'Arrow', 13, 15, facing=(1, 0))
  spawn(env, mods, 'Cow', 15, 17, health=2); spawn(env, mods, 'Arrow', 12, 17, facing=(1, 0))
  spawn(env, mods, 'Arrow', 12, 19, facing=(1, 0)); spawn(env, mods, 'Arrow', 16, 19, facing=(-1, 0))
  spawn(env, mods, 'Zombie', 15, 21, health=2, cooldown=9); spawn(env, mods, 'Arrow', 15, 23, facing=(0, -1))
  return [NOOP] * 12


def d_zombie_vs_sleeper(env, mods, rs):
  """A zombie hits a sleeping player for 7 (objects.py:305-311); the player wakes at its NEXT update
  (Q10); cooldown 5."""
  flatten(env, 4, 4, 17, 17)
  teleport(env, 10, 10, (0, 1))
  give(env, energy=2, health=9)
  env._player.sleeping = True
  spawn(env, mods, 'Zombie', 10, 11, cooldown=1)
  spawn(env, mods, 'Zombie', 9, 10, cooldown=4)
  return [SLEEP, SLEEP, SLEEP, NOOP, DO, DO, DO, SLEEP, SLEEP, SLEEP, SLEEP, SLEEP]


def d_dying_mobs(env, mods, rs):
  """Mobs at health <= 0 remove themselves and KEEP executing their update (Q3): they still draw,
  a zombie still hits, a skeleton still shoots; a hit on a mob that is already at 0 counts (Q5)."""
  flatten(env, 2, 2, 19, 19)
  teleport(env, 10, 10, (0, 1))
  give(env, health=9, wood_sword=1)
  spawn(env, mods, 'Zombie', 10, 11, health=0, cooldown=0)
  spawn(env, mods, 'Zombie', 11, 10, health=1, cooldown=0)
  spawn(env, mods, 'Skeleton', 10, 6, health=0, reload=0)
  spawn(env, mods, 'Skeleton', 6, 10, health=1, reload=0)
  spawn(env, mods, 'Cow', 9, 10, health=0)
  spawn(env, mods, 'Cow', 10, 9, health=1)
  w = env._world
  w[9, 9] = 'stone'; w[11, 9] = 'stone'; w[10, 8] = 'stone'  # the cow above cannot walk away
  return [DO, RIGHT, DO, DO, UP, DO, DO, LEFT, DO, DO, DOWN, DO, DO, NOOP, NOOP]


def d_skeleton_pen(env, mods, rs):
  """Skeletons that cannot flee (walled in) are fought in melee: defeat_skeleton, arrows shot at
  point-blank range hit the player (objects.py:203-206,327-351)."""
  flatten(env, 4, 4, 17, 17, 'path')
  teleport(env, 10, 10, (0, 1))
  give(env, health=9, iron_sword=1)
  spawn(env, mods, 'Skeleton', 10, 11, health=3, reload=0)
  spawn(env, mods, 'Skeleton', 9, 10, health=0, reload=0)
  spawn(env, mods, 'Skeleton', 10, 8, health=3, reload=2)
  w = env._world
  for x, y in ((9, 11), (11, 11), (10, 12), (8, 10), (9, 9), (9, 11), (9, 8), (11, 8), (10, 7)):
    w[x, y] = 'stone'
  return [NOOP, NOOP, DO, LEFT, DO, UP, NOOP, NOOP, NOOP, UP, DO, DO, NOOP]


def d_out_of_radius(env, mods, rs):
  """Objects at Manhattan distance >= 2*max(view) are frozen and draw nothing (Q1, env.py:86-89);
  a dead mob out there lingers until the player comes close (Q4)."""
  flatten(env, 0, 0, 64, 30)
  teleport(env, 5, 10, (1, 0))
  spawn(env, mods, 'Cow', 5 + 17, 10, health=0)
  spawn(env, mods, 'Cow', 5 + 18, 10, health=0)
  spawn(env, mods, 'Cow', 5 + 19, 10, health=0)
  spawn(env, mods, 'Zombie', 5 + 10, 10 + 7)
  spawn(env, mods, 'Zombie', 5 + 10, 10 + 8)
  spawn(env, mods, 'Zombie', 5 + 10, 10 + 9)
  spawn(env, mods, 'Arrow', 5 + 20, 12, facing=(1, 0))
  spawn(env, mods, 'Plant', 5 + 18, 14, grown=299)
  return [NOOP, NOOP, RIGHT, RIGHT, RIGHT, NOOP, LEFT, LEFT, LEFT, LEFT, NOOP, RIGHT, RIGHT]


def d_skeletons(env, mods, rs):
  """Skeletons at every range band around the player in tunnels: flee (<= 3), shoot (<= 5, reload),
  approach (<= 8), wander (objects.py:327-351); arrows spawn only into free arrow-walkable cells."""
  flatten(env, 0, 0, 40, 40, 'path')
  teleport(env, 20, 20, (0, 1))
  for dx, dy in ((2, 0), (-3, 0), (0, 4), (0, -5), (4, 1), (-2, 3), (6, 0), (0, -8), (9, 0), (3, 3)):
    spawn(env, mods, 'Skeleton', 20 + dx, 20 + dy, reload=int(rs.randint(0, 3)))
  env._world[20, 17] = 'stone'
  env._world[20, 23] = 'water'
  return [NOOP] * 10 + [LEFT, LEFT, UP, UP, NOOP, NOOP, DO, DO] + [NOOP] * 12


def d_sleep_cycle(env, mods, rs):
  """Falling asleep needs energy < 9 (Q11); asleep, the action is forced to sleep; waking up at full
  energy grants wake_up, here together with collect_wood in the same step (reward +1 once, Q9).
  Runs through nightfall: night noise + sleep filter in the renderer (engine.py:183-211)."""
  flatten(env, 6, 6, 15, 15)
  teleport(env, 10, 10, (0, 1))
  env._world[10, 11] = 'tree'
  give(env, energy=7)
  env._player._fatigue = -9
  set_step(env, 130)
  return [SLEEP] + [DO] * 40


def d_starve(env, mods, rs):
  """Necessities at zero: recover runs down, health drops one at a time, death at 0
  (objects.py:133-167)."""
  flatten(env, 6, 6, 15, 15)
  teleport(env, 10, 10, (0, 1))
  give(env, food=0, drink=1, energy=0, health=2)
  p = env._player
  p._recover, p._thirst, p._hunger, p._fatigue = -14.0, 20.0, 25.0, 30
  return [NOOP, LEFT, NOOP, SLEEP] + [NOOP] * 40


def d_regen_and_clamp(env, mods, rs):
  """Health regeneration at recover > 25, inventory clamped to 9 while achievements keep counting
  (objects.py:122-127)."""
  flatten(env, 6, 6, 15, 15)
  teleport(env, 10, 10, (0, 1))
  w = env._world
  w[10, 11] = 'tree'; w[11, 10] = 'water'
  give(env, wood=9, drink=9, health=5)
  env._player._recover = 24.0
  return [DO, DO, NOOP, RIGHT, DO, DO, NOOP]


def d_length_end(env, mods, rs):
  """Truncation: done when step >= length (env.py:106-107) with the player alive."""
  flatten(env, 6, 6, 15, 15)
  teleport(env, 10, 10, (0, 1))
  set_step(env, env._length - 3)
  return [NOOP, LEFT, RIGHT, NOOP, NOOP]


def d_balance_day(env, mods, rs):
  """Daylight balance ticks (env.py:141-179): crowded zombie / cow chunks despawn, skeletons need
  tunnels, target_fn truncation (Q13)."""
  flatten(env, 0, 0, 36, 36)
  flatten(env, 24, 0, 36, 12, 'path')
  teleport(env, 18, 18, (0, 1))
  for k in range(9):
    spawn(env, mods, 'Zombie', 1 + k, 2, cooldown=5)
    spawn(env, mods, 'Cow', 13 + k, 14)
  for k in range(5):
    spawn(env, mods, 'Skeleton', 25 + 2 * k, 5, reload=4)
  set_step(env, 8)
  return [NOOP] * 45


def d_balance_night(env, mods, rs):
  """Night balance: zombies spawn on grass in the dark (p 0.3 per tick and chunk), not next to the
  player (env.py:163-172)."""
  flatten(env, 0, 0, 48, 48)
  flatten(env, 36, 36, 48, 48, 'path')
  teleport(env, 20, 19, (0, 1))
  for cx in range(4):
    for cy in range(4):
      spawn(env, mods, 'Plant', cx * 12 + 6, cy * 12 + 6, grown=10)  # touches every chunk
  set_step(env, 188)
  return [NOOP, LEFT, RIGHT, UP, DOWN] * 10


def d_many_objects(env, mods, rs):
  """More than 128 slots: the ballot loop of the tick runs several rounds, arrows keep appending
  slots until the arena is compacted (engine.py:54-55; DESIGN.md section 1)."""
  flatten(env, 0, 0, 40, 40, 'path')
  teleport(env, 20, 20, (0, 1))
  n = 0
  for x in range(8, 33, 2):
    for y in range(8, 33, 3):
      if abs(x - 20) + abs(y - 20) < 3:
        continue
      kind = ('Cow', 'Skeleton', 'Cow', 'Zombie')[n % 4]
      attrs = dict(reload=0) if kind == 'Skeleton' else (dict(cooldown=5) if kind == 'Zombie' else {})
      spawn(env, mods, kind, x, y, **attrs)
      n += 1
  for x, y in ((19, 20), (21, 20), (20, 19), (20, 21)):  # a stone pen keeps the player alive
    env._world[x, y] = 'stone'
  return [NOOP] * 40


def d_double_unlock(env, mods, rs):
  """Two achievements in one step pay +1 once (Q9, env.py:99-104); a repeat pays nothing."""
  flatten(env, 6, 6, 15, 15)
  teleport(env, 10, 10, (0, 1))
  env._world[10, 11] = 'tree'
  give(env, energy=9)
  env._player.sleeping = True
  return [DO, DO, DO, NOOP]


DIRECTED = [
    ('craft_chain', d_craft_chain), ('gated_collects_fail', d_gated_collects_fail),
    ('edge_x0', _edge(0, 10, (-1, 0))), ('edge_y0', _edge(10, 0, (0, -1))),
    ('edge_origin', _edge(0, 0, (-1, 0))), ('edge_max', _edge(-1, -1, (1, 0))),
    ('edge_xmax', _edge(-1, 10, (1, 0))), ('lava_walk', d_lava_walk), ('plants', d_plants),
    ('sapling_luck', d_sapling_luck), ('water_lava_stone', d_water_lava_stone), ('arrows', d_arrows),
    ('zombie_vs_sleeper', d_zombie_vs_sleeper), ('dying_mobs', d_dying_mobs), ('skeleton_pen', d_skeleton_pen),
    ('out_of_radius', d_out_of_radius), ('skeletons', d_skeletons), ('sleep_cycle', d_sleep_cycle),
    ('starve', d_starve), ('regen_and_clamp', d_regen_and_clamp), ('length_end', d_length_end),
    ('balance_day', d_balance_day), ('balance_night', d_balance_night),
    ('many_objects', d_many_objects), ('double_unlock', d_double_unlock)]
