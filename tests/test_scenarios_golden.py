"""Corner-case scenarios recorded from the UNMODIFIED reference (tools/make_scenarios.py ->
tests/golden/scenarios/*.npz): states that random rollouts rarely reach -- crafting at map edges,
lava, dying mobs that still act, arrows against everything, sleep / wake, starvation, balance
ticks, > 128 slots ... (tests/scenario_util.py lists them with the reference lines they exercise).

All K scenarios of a group are loaded as ONE batch of K envs and stepped together; every step is
compared bit for bit with what the reference did: canonical state digests, the player vector,
reward, done, observation.  CPU: the device headers compiled for the host (tests/hostsim).
`-m gpu`: the CUDA library through crafter_b200.Env / the C ABI."""
import pathlib
import zlib

import numpy as np
import pytest

from oracle import canon
from tests import scenario_util as su

SCEN = pathlib.Path(__file__).resolve().parent / 'golden' / 'scenarios'
GROUPS = sorted(p.stem for p in SCEN.glob('*.npz'))


def to_numpy(x):
  return x.detach().cpu().numpy() if hasattr(x, 'detach') else np.asarray(x)


def replay_group(group, make_env, load, z=None):
  """z: the fixture's members (default: tests/golden/scenarios/<group>.npz)."""
  z = np.load(SCEN / f'{group}.npz') if z is None else z
  K = int(z['meta_K'])
  names = [str(n) for n in z['meta_names']]
  kwargs = dict(area=tuple(int(v) for v in z['meta_area']), view=tuple(int(v) for v in z['meta_view']),
                size=tuple(int(v) for v in z['meta_size']), length=int(z['meta_length']))
  env = make_env(num_envs=K, seed=int(z['meta_seed0']), auto_reset=False, **kwargs)
  env.reset()
  g = lambda i, k: z[f's{i}_{k}']
  for i in range(K):
    st = {k: g(i, k) for k in canon.KEYS}
    step, episode, world_seed = (int(v) for v in g(i, 'extras'))
    raw = su.raw_arrays(st, dict(step=step, episode=episode, world_seed=world_seed), kwargs['area'],
                        env.state['ents'].shape[1])
    load(env.state, i, raw)
  if hasattr(env, 'recount'):
    env.recount()  # the terrain was written behind the implementation's back
  obs = to_numpy(env.render())
  for i in range(K):
    st = {k: g(i, k) for k in canon.KEYS}
    assert canon.diff(st, env.snapshot(i)) is None, (group, names[i], 'load')
    assert zlib.crc32(np.ascontiguousarray(obs[i]).tobytes()) == int(g(i, 'init_obs_crc')), (
        group, names[i], 'render after load')
  n = [len(g(i, 'actions')) for i in range(K)]
  compared = 0
  for t in range(max(n)):
    actions = np.array([g(i, 'actions')[t] if t < n[i] else 0 for i in range(K)], np.int32)
    obs, reward, done = env.step(actions)[:3]
    obs, reward, done = to_numpy(obs), to_numpy(reward), to_numpy(done).astype(bool)
    for i in range(K):
      if t >= n[i]:
        continue  # this scenario has ended (the reference env was done); its env idles on
      where = (group, names[i], t, int(actions[i]))
      snap = env.snapshot(i)
      ref_player = g(i, 'player_t')[t]
      assert (snap['player'] == ref_player).all(), (
          where, 'player', np.flatnonzero(snap['player'] != ref_player).tolist(),
          snap['player'][snap['player'] != ref_player].tolist(),
          ref_player[snap['player'] != ref_player].tolist())
      for k, v in canon.digest(snap).items():
        assert v == int(g(i, f'{k}_crc')[t]), (where, k)
      assert reward[i] == np.float32(g(i, 'reward')[t]), (where, 'reward', reward[i], g(i, 'reward')[t])
      assert bool(done[i]) == bool(g(i, 'done')[t]), (where, 'done')
      assert zlib.crc32(np.ascontiguousarray(obs[i]).tobytes()) == int(g(i, 'obs_crc')[t]), (where, 'obs')
      compared += 1
  assert compared == sum(n) and compared > 0
  return env


def test_fixtures_present():
  assert {'fuzz_default', 'fuzz_small', 'fuzz_big_view', 'directed_default', 'directed_short'} <= set(GROUPS)


def test_directed_scenarios_reach_their_corners():
  """The fixtures really contain what their names say (so a green replay means something)."""
  z = np.load(SCEN / 'directed_default.npz')
  names = [str(n) for n in z['meta_names']]
  ach = {n: z[f's{i}_player_t'][:, 16:38].max(0) for i, n in enumerate(names)}
  done = {n: bool(z[f's{i}_done'].any()) for i, n in enumerate(names)}
  A = canon_achievements()
  for a in ('make_wood_pickaxe', 'make_stone_pickaxe', 'make_iron_pickaxe', 'make_wood_sword',
            'make_stone_sword', 'make_iron_sword', 'collect_diamond', 'collect_iron', 'collect_coal',
            'collect_stone', 'place_stone', 'place_table', 'place_furnace'):
    assert ach['craft_chain'][A[a]] >= 1, a
  assert ach['craft_chain'][A['make_iron_sword']] == 2
  assert ach['gated_collects_fail'].sum() == 0
  for edge in ('edge_x0', 'edge_y0', 'edge_origin'):  # Q7: no crafting where x == 0 or y == 0
    assert ach[edge][[A['make_wood_pickaxe'], A['make_iron_sword']]].sum() == 0, edge
  assert ach['edge_max'][A['make_wood_pickaxe']] >= 1 and ach['edge_xmax'][A['make_iron_sword']] >= 1
  assert done['lava_walk'] and done['starve'] and done['length_end']
  assert ach['plants'][A['eat_plant']] >= 1 and ach['plants'][A['place_plant']] >= 1
  assert ach['sapling_luck'][A['collect_sapling']] >= 1
  assert ach['water_lava_stone'][A['collect_drink']] >= 1 and ach['water_lava_stone'][A['place_stone']] >= 2
  assert ach['dying_mobs'][A['defeat_zombie']] >= 2 and ach['dying_mobs'][A['eat_cow']] >= 1  # Q5
  assert ach['sleep_cycle'][A['wake_up']] >= 1 and ach['double_unlock'][A['wake_up']] == 1
  i = names.index('double_unlock')  # Q9: wake_up + collect_wood in one step pay +1 once
  assert z[f's{i}_reward'][0] == 1.0 and z[f's{i}_reward'][1] == 0.0
  i = names.index('zombie_vs_sleeper')  # 7 damage to a sleeper
  assert (np.diff(np.concatenate([[9], z[f's{i}_player_t'][:, 0]])) == -7).any()
  i = names.index('many_objects')
  assert len(z[f's{i}_objs']) > 100


def canon_achievements():
  from crafter_b200 import rules
  return {a: k for k, a in enumerate(rules.ACHIEVEMENTS)}


@pytest.mark.parametrize('group', GROUPS)
def test_hostsim_replays_scenarios(group):
  from tests import hostsim_env
  replay_group(group, hostsim_env.HostSimEnv, su.load_numpy)


def test_hostsim_replays_scenarios_with_tiny_arenas():
  """Same fixtures with a 2-entry object-tile cache (per-pixel path of the renderer) and the smallest
  slot arena the largest scenario fits (order-preserving compaction while arrows keep appending)."""
  import functools
  from tests import hostsim_env
  replay_group('directed_default', functools.partial(hostsim_env.HostSimEnv, max_obj_tiles=2), su.load_numpy)
  env = replay_group('directed_default', functools.partial(hostsim_env.HostSimEnv, slot_capacity=192),
                     su.load_numpy)
  assert int(np.abs(env.state['pstate'][:, 14]).sum()) == 0  # no overflow bit


def make_cuda_env(**kwargs):
  import crafter_b200
  return crafter_b200.Env(**kwargs)


@pytest.mark.gpu
@pytest.mark.parametrize('group', GROUPS)
def test_cuda_replays_scenarios(group):
  replay_group(group, make_cuda_env, su.load_torch)


@pytest.mark.gpu
def test_cuda_replays_scenarios_generic_kernels_and_small_arena(monkeypatch):
  import functools
  env = replay_group('directed_default', functools.partial(make_cuda_env, slot_capacity=192), su.load_torch)
  assert int(env.state['pstate'][:, 14].abs().sum()) == 0
  monkeypatch.setenv('CRAFTER_B200_NO_SPECIALIZE', '1')
  replay_group('directed_default', make_cuda_env, su.load_torch)


@pytest.mark.parametrize('group', GROUPS)
def test_c_oracle_replays_scenarios(group):
  """The C restatement (the checker behind smoke() and the CPU baseline) on the same fixtures."""
  from oracle import oracle_env
  z = np.load(SCEN / f'{group}.npz')
  names = [str(n) for n in z['meta_names']]
  kwargs = dict(area=tuple(int(v) for v in z['meta_area']), view=tuple(int(v) for v in z['meta_view']),
                size=tuple(int(v) for v in z['meta_size']), length=int(z['meta_length']))
  for i, name in enumerate(names):
    g = lambda k: z[f's{i}_{k}']
    env = oracle_env.OracleEnv(seed=int(z['meta_seed0']) + i, **kwargs)
    env.reset()
    st = {k: g(k) for k in canon.KEYS}
    env.import_state(st, *(int(v) for v in g('extras')))
    assert canon.diff(st, env.export_state()) is None, (group, name, 'load')
    assert zlib.crc32(env.render().tobytes()) == int(g('init_obs_crc')), (group, name, 'render after load')
    for t, a in enumerate(g('actions')):
      obs, reward, done = env.step(int(a))
      snap = env.export_state()
      assert (snap['player'] == g('player_t')[t]).all(), (group, name, t, 'player')
      for k, v in canon.digest(snap).items():
        assert v == int(g(f'{k}_crc')[t]), (group, name, t, k)
      assert reward == g('reward')[t] and done == bool(g('done')[t]), (group, name, t, reward)
      assert zlib.crc32(obs.tobytes()) == int(g('obs_crc')[t]), (group, name, t, 'obs')
