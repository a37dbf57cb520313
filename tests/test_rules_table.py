"""The rule tables of data.yaml three ways: crafter_b200/rules.py (the restatement) == the reference's
data.yaml (stored parsed as tests/golden/data_yaml.json by tools/make_rules_golden.py), and the DEVICE code
(csrc/cr_update.h, csrc/cr_worldgen.h, compiled for the host) behaves as rules.py says, entry by
entry: every collect (tool gate, item, material left, the 10 % sapling draw), every place (cost,
allowed ground, result) and every make (cost, nearby table / furnace), the walkable set, the
inventory clamp and the initial inventory.  The scenario fixtures reach the same rules through whole
trajectories of the reference; this is the direct diff the literals never had."""
import json
import pathlib

import numpy as np
import pytest

from crafter_b200 import rules
from tests import hostsim_env

DATA = pathlib.Path(__file__).resolve().parent / 'golden' / 'data_yaml.json'
MAT = {name: i + 1 for i, name in enumerate(rules.MATERIALS)}
ITEM = {name: i for i, name in enumerate(rules.ITEMS)}
ACT = {name: i for i, name in enumerate(rules.ACTIONS)}
ACH = {name: i for i, name in enumerate(rules.ACHIEVEMENTS)}


def test_rules_py_equals_data_yaml():
  d = json.loads(DATA.read_text())
  assert d['actions'] == rules.ACTIONS and d['materials'] == rules.MATERIALS
  assert d['achievements'] == rules.ACHIEVEMENTS
  assert list(d['items']) == rules.ITEMS  # order is semantics (engine.py:230,238)
  assert sorted(d['walkable']) == sorted(rules.WALKABLE)
  for name, spec in d['items'].items():
    assert spec['max'] == rules.ITEM_MAX and spec['initial'] == rules.ITEM_INITIAL.get(name, 0), name
  assert set(d['collect']) == set(rules.COLLECT)
  for name, spec in d['collect'].items():
    tool, item, leaves, prob = rules.COLLECT[name]
    assert spec['require'] == ({tool: 1} if tool else {}) and spec['receive'] == {item: 1}, name
    assert spec['leaves'] == leaves and spec.get('probability', 1.0) == prob, name
  assert set(d['place']) == set(rules.PLACE)
  for name, spec in d['place'].items():
    item, amount, where, kind = rules.PLACE[name]
    assert spec['uses'] == {item: amount} and sorted(spec['where']) == sorted(where) and spec['type'] == kind, name
  assert set(d['make']) == set(rules.MAKE)
  for name, spec in d['make'].items():
    uses, nearby = rules.MAKE[name]
    assert spec['uses'] == uses and sorted(spec['nearby']) == sorted(nearby) and spec['gives'] == 1, name


def fresh(seed=3):
  """One env on a tiny all-grass map, the player in the middle facing down, nothing else alive."""
  env = hostsim_env.HostSimEnv(num_envs=1, area=(9, 9), seed=seed, length=100000)
  env.reset()
  s = env.state
  s['mat'][0, :] = MAT['grass']
  s['objmap'][0, :] = 0
  s['objmap'][0, 4 * 9 + 4] = 1
  ents = s['ents'][0].view(np.uint8).reshape(-1, 8)
  ents[2:, 0] = 0  # tombstone every creature
  s['pstate'][0, 8] = 2
  env.recount()
  return env


def front(env, material):
  env.state['mat'][0, 4 * 9 + 5] = MAT[material]  # the cell below the player (facing down)
  env.recount()


def inv(env, name):
  return int(env.state['inventory'][0, ITEM[name]])


def test_initial_inventory_and_clamp():
  env = fresh()
  for name in rules.ITEMS:
    assert inv(env, name) == rules.ITEM_INITIAL.get(name, 0), name
  env.set_inventory({'wood': 9})
  front(env, 'tree')
  env.step(np.array([ACT['do']], np.int32))
  assert inv(env, 'wood') == rules.ITEM_MAX  # objects.py:126-128


@pytest.mark.parametrize('material', list(rules.COLLECT))
def test_collect_entry(material):
  tool, item, leaves, prob = rules.COLLECT[material]
  ach = {'wood': 'collect_wood', 'stone': 'collect_stone', 'coal': 'collect_coal', 'iron': 'collect_iron',
         'diamond': 'collect_diamond', 'drink': 'collect_drink', 'sapling': 'collect_sapling'}[item]
  if tool:  # without the tool: nothing happens, the material stays
    env = fresh()
    front(env, material)
    env.step(np.array([ACT['do']], np.int32))
    assert inv(env, item) == rules.ITEM_INITIAL.get(item, 0) and env.state['mat'][0, 4 * 9 + 5] == MAT[material]
    lesser = {'stone_pickaxe': 'wood_pickaxe', 'iron_pickaxe': 'stone_pickaxe'}.get(tool)
    if lesser:  # the next lower tool does not do either
      env.set_inventory({lesser: 1})
      env.step(np.array([ACT['do']], np.int32))
      assert env.state['mat'][0, 4 * 9 + 5] == MAT[material]
  got, trials = 0, 400 if prob < 1 else 3
  for trial in range(trials):
    env = fresh(seed=trial)
    if tool:
      env.set_inventory({tool: 1})
    if item == 'drink':
      env.set_inventory({'drink': 5})
    front(env, material)
    before = inv(env, item)
    env.step(np.array([ACT['do']], np.int32))
    assert env.state['mat'][0, 4 * 9 + 5] == MAT[leaves], (material, leaves)
    gained = inv(env, item) - before
    assert gained in (0, 1) and int(env.state['achievements'][0, ACH[ach]]) == gained
    got += gained
  if prob < 1:
    assert abs(got / trials - prob) < 4 * (prob * (1 - prob) / trials) ** 0.5, got / trials  # 4 sigma
  else:
    assert got == trials


@pytest.mark.parametrize('name', list(rules.PLACE))
def test_place_entry(name):
  item, amount, where, kind = rules.PLACE[name]
  action = np.array([ACT[f'place_{name}']], np.int32)
  for ground in rules.MATERIALS:
    env = fresh()
    env.set_inventory({item: amount})
    front(env, ground)
    env.step(action)
    placed = ground in where
    assert inv(env, item) == (0 if placed else amount), (name, ground)
    assert int(env.state['achievements'][0, ACH[f'place_{name}']]) == int(placed)
    if kind == 'material':
      assert env.state['mat'][0, 4 * 9 + 5] == MAT[name if placed else ground], (name, ground)
    else:  # a Plant object on unchanged ground
      assert env.state['mat'][0, 4 * 9 + 5] == MAT[ground]
      assert (env.state['objmap'][0, 4 * 9 + 5] != 0) == placed
  env = fresh()  # one item short: nothing happens
  env.set_inventory({item: amount - 1})
  front(env, where[0])
  env.step(action)
  assert inv(env, item) == amount - 1 and env.state['mat'][0, 4 * 9 + 5] == MAT[where[0]]


@pytest.mark.parametrize('name', list(rules.MAKE))
def test_make_entry(name):
  uses, nearby = rules.MAKE[name]
  action = np.array([ACT[f'make_{name}']], np.int32)

  def attempt(have, near):
    env = fresh()
    env.set_inventory(have)
    for k, m in enumerate(near):
      env.state['mat'][0, (3 + k) * 9 + 3] = MAT[m]  # diagonal neighbours of the player at (4, 4)
    env.recount()
    env.step(action)
    return env

  env = attempt(uses, nearby)
  assert inv(env, name) == 1 and all(inv(env, k) == 0 for k in uses)
  assert int(env.state['achievements'][0, ACH[f'make_{name}']]) == 1
  for missing in nearby:  # each nearby requirement on its own
    env = attempt(uses, [m for m in nearby if m != missing])
    assert inv(env, name) == 0 and all(inv(env, k) == v for k, v in uses.items())
  for short in uses:  # each ingredient on its own
    env = attempt({k: v - (k == short) for k, v in uses.items()}, nearby)
    assert inv(env, name) == 0


def test_walkable_set():
  for ground in rules.MATERIALS:
    env = fresh()
    front(env, ground)
    env.step(np.array([ACT['move_down']], np.int32))
    moved = int(env.state['pstate'][0, 13]) == 5
    assert moved == (ground in rules.WALKABLE or ground == 'lava'), ground  # the player may walk into lava (objects.py:95-97)
