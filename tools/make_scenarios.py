"""Generate tests/golden/scenarios/*.npz from the UNMODIFIED reference (build container only).

Random rollouts (tests/golden/*.npz) rarely reach the corners of the rules, so these fixtures start
from states built inside live reference envs through the reference's own World / object API
(tests/scenario_util.py): a perturbation fuzz and one directed scenario per rule corner.  Each
scenario stores the canonical start state (oracle/canon.py), the actions, and per step the digests
of the canonical state, reward, done and the observation digest -- all produced by the reference
under oracle/ref_harness.py.  tests/test_scenarios_golden.py replays them through the host-sim on
CPU and through the CUDA library (C ABI) on the GPU box.

    python tools/make_scenarios.py            # writes every group in GROUPS and PERTURBED
    python tools/make_scenarios.py perturbed  # only tests/golden/perturbed/
"""
import pathlib
import sys
import zlib

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

from oracle import canon  # noqa: E402
from oracle import ref_harness as rh  # noqa: E402
from tests import scenario_util as su  # noqa: E402

GROUPS = {
    # name: (env kwargs, kind, count / None, base seed)
    'fuzz_default': (dict(), 'fuzz', 40, 900),
    'fuzz_small': (dict(area=(24, 20)), 'fuzz', 30, 900),
    'fuzz_big_view': (dict(view=(15, 15), size=(128, 128)), 'fuzz', 8, 1900),
    'fuzz_big_area': (dict(area=(256, 256)), 'fuzz', 6, 2900),
    'directed_default': (dict(), 'directed', None, 3000),
    'directed_short': (dict(length=300, area=(48, 56), view=(7, 9), size=(70, 72)), 'directed', None, 4000),
}
FUZZ_STEPS = 45
# The perturbation stream tests/test_scenarios_vs_reference.py replays from tests/golden/perturbed/
# (random stream 4711, world seeds 5000 + round): name -> (env kwargs, rounds, steps per round)
PERTURBED = {
    'default': (dict(), 40, 45),
    'small': (dict(area=(24, 20)), 30, 40),
}


def record(env, actions):
  st0 = rh.export_state(env)
  out = dict(mat=st0['mat'], objs=st0['objs'], player=st0['player'], touched=st0['touched'],
             extras=np.array([env._step, env._episode, env._world.random.seed], np.int64),
             init_obs_crc=np.array(zlib.crc32(env.render().tobytes()), np.int64))
  rec = dict(reward=[], done=[], obs_crc=[], player_t=[])
  for k in canon.KEYS:
    rec[k + '_crc'] = []
  done_actions = []
  obs = None
  for a in actions:
    obs, reward, done, info = env.step(int(a))
    st = rh.export_state(env)
    done_actions.append(int(a))
    rec['reward'].append(reward)
    rec['done'].append(done)
    rec['obs_crc'].append(zlib.crc32(obs.tobytes()))
    rec['player_t'].append(st['player'])
    for k, v in canon.digest(st).items():
      rec[k + '_crc'].append(v)
    if done:
      break
  out['actions'] = np.array(done_actions, np.int32)
  out['reward'] = np.array(rec['reward'], np.float64)
  out['done'] = np.array(rec['done'], bool)
  out['obs_crc'] = np.array(rec['obs_crc'], np.int64)
  out['player_t'] = np.array(rec['player_t'], np.int64).reshape(-1, 49)
  for k in canon.KEYS:
    out[k + '_crc'] = np.array(rec[k + '_crc'], np.int64)
  out['obs_last'] = obs
  return out


def build(kwargs, kind, count, seed0, stream=2024, steps=FUZZ_STEPS):
  mods = rh.load()
  scenarios, names = [], []
  if kind == 'fuzz':
    rs = np.random.RandomState(stream)
    for r in range(count):
      env = rh.make_env(seed0 + r, **kwargs)
      env.reset()
      su.perturb(env, rs, mods)
      scenarios.append(record(env, su.fuzz_actions(rs, steps)))
      names.append(f'fuzz{r}')
  else:
    for r, (name, fn) in enumerate(su.DIRECTED):
      env = rh.make_env(seed0 + r, **kwargs)
      env.reset()
      rs = np.random.RandomState(77 + r)
      actions = fn(env, mods, rs)
      scenarios.append(record(env, actions))
      names.append(name)
  return names, scenarios


def main(groups):
  for g in groups:
    if g == 'perturbed':
      for name, (kwargs, count, steps) in PERTURBED.items():
        names, scenarios = build(kwargs, 'fuzz', count, 5000, stream=4711, steps=steps)
        for s in scenarios:
          del s['obs_last']  # no replay reads it, and it would be half of the file
        save(ROOT / 'tests' / 'golden' / 'perturbed' / f'{name}.npz', kwargs, 5000, names, scenarios, packed=True)
    else:
      kwargs, kind, count, seed0 = GROUPS[g]
      names, scenarios = build(kwargs, kind, count, seed0)
      save(ROOT / 'tests' / 'golden' / 'scenarios' / f'{g}.npz', kwargs, seed0, names, scenarios)


def save(path, kwargs, seed0, names, scenarios, packed=False):
  blob = dict(
      meta_area=np.array(kwargs.get('area', (64, 64))), meta_view=np.array(kwargs.get('view', (9, 9))),
      meta_size=np.array(kwargs.get('size', (64, 64))), meta_length=np.array(kwargs.get('length', 10000)),
      meta_seed0=np.array(seed0), meta_K=np.array(len(scenarios)), meta_names=np.array(names))
  ach, steps, deaths = 0, 0, 0
  for i, s in enumerate(scenarios):
    for k, v in s.items():
      blob[f's{i}_{k}'] = v
    ach |= int(s['player_t'][:, 16:38].max(0).astype(bool) @ (1 << np.arange(22)))
    steps += len(s['actions'])
    deaths += int(s['done'].any())
  path.parent.mkdir(parents=True, exist_ok=True)
  np.savez_compressed(path, **(su.pack(blob) if packed else blob))
  print(f'{path.stem}: {len(scenarios)} scenarios, {steps} steps, {deaths} ended, '
        f'{bin(ach).count("1")}/22 achievements touched, {path.stat().st_size / 1024:.0f} KiB')


if __name__ == '__main__':
  main(sys.argv[1:] or list(GROUPS) + ['perturbed'])
