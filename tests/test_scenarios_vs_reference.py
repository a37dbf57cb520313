"""Perturbation fuzz recorded from the UNMODIFIED reference (tools/make_scenarios.py perturbed ->
tests/golden/perturbed/*.npz): random-policy trajectories rarely reach the corner cases of the rules
(crafting at the map edge, lava, dying mobs that still act, arrows hitting things, ripe plants,
full inventories ...), so the recorder teleported the player, rewrote terrain, spawned creatures
with odd attributes and set inventories *inside the reference env through its own API*, then
stepped it with random actions.  This test loads the very same canonical states into the device
logic (host-sim build of csrc/cr_*.h) and steps it with the recorded actions, comparing the full
integer state, reward, done and the observation each step with what the reference did."""
import pathlib

import numpy as np
import pytest

from tests import hostsim_env
from tests import scenario_util as su
from tests.test_scenarios_golden import replay_group

PERTURBED = pathlib.Path(__file__).resolve().parent / 'golden' / 'perturbed'


@pytest.mark.parametrize('geometry', [dict(), dict(area=(24, 20))])
def test_perturbed_states_step_like_the_reference(geometry):
  name = 'small' if geometry else 'default'
  env = replay_group(name, hostsim_env.HostSimEnv, su.load_numpy, su.unpack(np.load(PERTURBED / f'{name}.npz')))
  assert env.area == geometry.get('area', (64, 64))
