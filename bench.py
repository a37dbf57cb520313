"""bench.py -- env steps/sec of a batched random-policy Crafter rollout on N B200s (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config NAME]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one tick of every env of the batch.  `--config default` is BASELINE.json configs[1]
(`num_envs=4096, area=(64,64), view=(9,9)` per GPU; configs[2] is 8 x 4096 with no collective on the
step path, i.e. weak scaling); `area256` is configs[3] (1024 envs on 256 x 256 maps) and `view15`
configs[4] (4096 envs, 128 x 128 observations of a 15 x 15 view).  Actions come from a pre-generated
synthetic (T, B) int32 tensor; finished episodes are regenerated inside the step.

The metric is a steady-state quantity (the reference's protocol, crafter/run_random.py:36-43, is a
wall clock around a loop WITH resets), so whatever --warmup / --steps say the batch is first rolled
forward `--preroll` untimed steps (default 1000, about 0.1 s): the episodes of a fresh batch are
synchronised (all daytime, no death before step 23, every env balancing on the same steps) and only
desynchronise through their first few resets (mean episode length 168).  The `regime` block of the
JSON line says what the timed window actually contained: night fraction, resets per step, the
fraction of envs balancing, worlds generated.

Timing: W untimed steps, then K steps; each timed step is bracketed by CUDA events on the env's
stream with a 256 MiB L2 flush between steps (outside the events); ms_per_step is the mean of those
K device durations, max over ranks.  `e2e` is the same metric through `cr_step_host` with pinned
HOST buffers (H2D actions, D2H reward/done, stream sync, every step), timed per rank by the host
clock between two stream synchronisations, max over ranks AFTERWARDS (no collective inside the
window).  `roofline` / `kernels`: per-kernel device durations measured INSIDE the step graph by
event-record nodes around every kernel (CRAFTER_B200_TIMING=2) over the same state.  One JSON line
on rank 0.
"""
import argparse
import ctypes
import json
import os
import pathlib
import subprocess
import sys
import threading
import time

ROOT = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = 'env_steps_per_sec_random_policy'
UNIT = 'env-steps/s'
CONFIGS = {
    'default': dict(num_envs=4096, area=(64, 64), view=(9, 9), size=(64, 64), tag='BASELINE.json configs[1]'),
    'area256': dict(num_envs=1024, area=(256, 256), view=(9, 9), size=(64, 64), tag='BASELINE.json configs[3]'),
    'view15': dict(num_envs=4096, area=(64, 64), view=(15, 15), size=(128, 128), tag='BASELINE.json configs[4]'),
}
KERNEL_NAMES = ['k_update', 'k_install', 'k_render', 'k_seed', 'k_wg_mat', 'k_wg_obj', 'k_seed_ahead', 'k_post']


def env_kwargs(cfg):
  return {k: cfg[k] for k in ('num_envs', 'area', 'view', 'size')}


def render_bytes_per_env(cfg):
  """SURVEY.md section 8(d): algorithmic bytes per env-step of the render kernel = W*H*3 obs store +
  3*vx*(vy-rows) window read (u8 mat + u16 slot) + 256 B of player / entity records."""
  item_rows = -(-16 // cfg['view'][0])
  return cfg['size'][0] * cfg['size'][1] * 3 + 3 * cfg['view'][0] * (cfg['view'][1] - item_rows) + 256


def workload_config(name, n_gpus, preroll):
  c = CONFIGS[name]
  return {
      'workload': f'crafter random-policy rollout, num_envs={c["num_envs"]} per GPU, area={c["area"]}, '
                  f'view={c["view"]}, size={c["size"]}, length=10000, auto-reset ({c["tag"]})',
      'global_num_envs': c['num_envs'] * n_gpus,
      'parallelism': f'env-batch sharded x{n_gpus}, no collective on the step path',
      'l2': 'flushed between timed steps (256 MiB memset outside the per-step CUDA events)',
      'preroll_steps': preroll,
  }


class ClockSampler:
  """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
  Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
       'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
       'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

  def __init__(self, index):
    self.index, self.lines, self.proc = index, [], None

  def start(self):
    try:
      self.proc = subprocess.Popen(
          ['nvidia-smi', f'--id={self.index}', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
           '-lms', '50'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      threading.Thread(target=self._read, daemon=True).start()
    except Exception:
      self.proc = None

  def _read(self):
    for line in self.proc.stdout:
      self.lines.append(line.strip())

  def stop(self):
    if self.proc:
      time.sleep(0.15)
      self.proc.terminate()
    sm, mx, reasons = [], [], set()
    for line in self.lines:
      p = [x.strip() for x in line.split(',')]
      if len(p) < 9:
        continue
      try:
        sm.append(float(p[1])); mx.append(float(p[2]))
      except ValueError:
        continue
      for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown',
                          'sw_power_cap'), p[5:9]):
        if v.lower().startswith('active'):
          reasons.add(name)
    sm.sort()
    return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None,
            'reasons': sorted(reasons), 'samples': len(sm)}


# ---- CPU legs: the oracle port of the reference env on the host cores -----------------------------
def _oracle_batch(cfg, cores, preroll):
  """A bounded sample of the workload (32 envs per host thread), rolled forward to the same
  desynchronised steady state as the GPU batch before anything is timed."""
  import numpy as np
  from oracle import oracle_env
  n_env = min(cfg['num_envs'], 32 * cores)
  batch = oracle_env.OracleBatch(n_env, cores, seed=0, area=cfg['area'], view=cfg['view'], size=cfg['size'])
  batch.reset()
  rs = np.random.RandomState(0)
  t0 = time.perf_counter()
  for _ in range(preroll):
    batch.step(rs.randint(0, 17, n_env))
    if time.perf_counter() - t0 > 60:  # slow hosts: a shorter pre-roll is said in `sample`
      break
  return batch, rs, n_env


def cpu_baseline(cfg, cores, preroll, budget_s=10.0):
  """The oracle port (oracle/crafter_oracle.c: the reference's algorithm restated in C, pinned to
  the unmodified reference by tests/golden) on the host cores: same workload shape, bounded sample."""
  batch, rs, n_env = _oracle_batch(cfg, cores, preroll)
  t0, n = time.perf_counter(), 0
  while time.perf_counter() - t0 < budget_s:
    batch.step(rs.randint(0, 17, n_env))
    n += 1
  dt = time.perf_counter() - t0
  return {'value': n * n_env / dt, 'unit': UNIT, 'cores': cores, 'kind': 'port',
          'sample': f'{n} batched ticks of {n_env} of the {cfg["num_envs"]} envs (step + render + '
                    f'reset-on-done) after a {preroll}-step pre-roll, C oracle port, {cores} threads, {dt:.1f} s'}


def run_reference(args, rank, world):
  """--impl reference: the reference's CPU implementation of the path on the host cores.  The
  reference is pure Python and cannot travel to the GPU box, so this times the oracle port."""
  if rank != 0:
    return
  cfg = CONFIGS[args.config]
  cores = os.cpu_count() or 1
  batch, rs, n_env = _oracle_batch(cfg, cores, args.preroll)
  for _ in range(args.warmup):
    batch.step(rs.randint(0, 17, n_env))
  t0 = time.perf_counter()
  for _ in range(args.steps):
    batch.step(rs.randint(0, 17, n_env))
  dt = time.perf_counter() - t0
  value = args.steps * n_env / dt
  sample = (f'each step = one tick of {n_env} of the {cfg["num_envs"]} envs (bounded sample) after a '
            f'{args.preroll}-step pre-roll, oracle C port of the reference env on {cores} host threads')
  print(json.dumps({
      'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus,
      'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * dt / args.steps,
      'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'int32/f64',
      'data': 'synthetic', 'config': workload_config(args.config, args.gpus, args.preroll),
      'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                       'sample': sample},
      'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}))


# ---- regime of a timed window ---------------------------------------------------------------------
def regime_probe(env):
  """Per-env step and episode counters (device tensors, cloned): two probes bracket a window."""
  ps = env.state['pstate']
  return ps[:, 9].clone(), ps[:, 10].clone()


def regime_block(before, after, steps):
  import torch
  out = {}
  for name, (step, _) in (('start', before), ('end', after)):
    phase = step % 300
    out[f'night_fraction_{name}'] = float(((phase >= 148) & (phase <= 272)).float().mean())
  out['balancing_fraction_end'] = float((after[0] % 10 == 0).float().mean())
  resets = int((after[1] - before[1]).sum())
  out['resets_per_step'] = resets / max(steps, 1)
  out['worlds_generated'] = resets
  out['mean_env_step_end'] = float(after[0].float().mean())
  return out


DUMP_BYTES = 60 * 10 ** 6  # what --dump-outputs writes in all stays below 64 MB, .npy headers included


def dump_outputs(directory, obs, reward, done, info):
  """What the last timed step returned, as float32 DIR/<name>.npy (every value is a small integer or a
  reward, so exactly): reward, done, inventory, achievements and player_pos of every env, and obs of
  every env when they fit, else of a fixed sample of envs (np.random.RandomState(0), ascending)."""
  import numpy as np
  import torch
  out = pathlib.Path(directory)
  out.mkdir(parents=True, exist_ok=True)
  arrays = dict(reward=reward, done=done, inventory=info['inventory'], achievements=info['achievements'],
                player_pos=info['player_pos'])
  B = obs.shape[0]
  n = min(B, (DUMP_BYTES - 4 * sum(a.numel() for a in arrays.values())) // (4 * obs[0].numel()))
  rows = np.sort(np.random.RandomState(0).choice(B, n, replace=False)) if n < B else np.arange(B)
  arrays['obs'] = obs[torch.as_tensor(rows, device=obs.device)]
  for name, a in arrays.items():
    np.save(out / f'{name}.npy', a.cpu().numpy().astype(np.float32))


def kernel_times(kwargs, seed, rank_offset, state_dict, actions, steps):
  """Per-kernel device durations INSIDE the step graph: a second handle created with
  CRAFTER_B200_TIMING=2 (event-record nodes around every kernel of the captured graph), loaded with
  the steady-state snapshot of the benchmarked batch and stepped with the same actions."""
  import crafter_b200
  old = os.environ.get('CRAFTER_B200_TIMING')
  os.environ['CRAFTER_B200_TIMING'] = '2'
  try:
    env = crafter_b200.Env(seed=seed, auto_reset=True, env_offset=rank_offset, **kwargs)
  finally:
    if old is None:
      os.environ.pop('CRAFTER_B200_TIMING', None)
    else:
      os.environ['CRAFTER_B200_TIMING'] = old
  env.reset()
  env.load_state_dict(state_dict)
  out = (ctypes.c_double * 8)()
  for t in range(10):
    env.step(actions[t % len(actions)])
  env._lib.cr_timing(env._handle, out)  # drop the warm-up
  for t in range(steps):
    env.step(actions[(10 + t) % len(actions)])
  n = env._lib.cr_timing(env._handle, out)
  times = {k: out[i] for i, k in enumerate(KERNEL_NAMES) if out[i] > 0}
  env.close()
  return n, times


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=2000)
  ap.add_argument('--warmup', type=int, default=200)
  ap.add_argument('--preroll', type=int, default=1000, help='untimed steps before the warm-up (steady state)')
  ap.add_argument('--config', default='default', choices=sorted(CONFIGS))
  ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
  ap.add_argument('--no-cpu-baseline', action='store_true')
  ap.add_argument('--dump-outputs', metavar='DIR',
                  help='write what the last timed step returned (rank 0) as DIR/<name>.npy, see dump_outputs')
  args = ap.parse_args()
  if args.steps < 1:
    ap.error('--steps must be at least 1')
  if args.dump_outputs and args.impl != 'ours':
    ap.error('--dump-outputs writes what the CUDA path returned; it needs --impl ours')
  args.warmup = max(args.warmup, 3)
  rank = int(os.environ.get('RANK', 0))
  local_rank = int(os.environ.get('LOCAL_RANK', 0))
  world = int(os.environ.get('WORLD_SIZE', 1))
  if args.impl == 'reference':
    return run_reference(args, rank, world)

  import torch
  import torch.distributed as dist
  import crafter_b200

  torch.cuda.set_device(local_rank)
  device = torch.device('cuda', local_rank)
  if world > 1:
    dist.init_process_group('nccl', device_id=device)
  assert world == args.gpus, f'--gpus {args.gpus} but WORLD_SIZE={world} (launch with torchrun)'

  cfg = CONFIGS[args.config]
  kwargs = env_kwargs(cfg)
  B, K, W = cfg['num_envs'], args.steps, args.warmup
  env = crafter_b200.Env(seed=0, auto_reset=True, env_offset=rank * B, device=device, **kwargs)
  T = 512
  gen = torch.Generator(device=device).manual_seed(1234 + rank)
  actions = torch.randint(0, 17, (T, B), generator=gen, device=device, dtype=torch.int32)
  flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)
  stream = env._stream
  env.reset()
  for t in range(args.preroll):  # to the desynchronised steady state, whatever W and K are
    env.step(actions[t % T])
  for t in range(W):
    env.step(actions[(args.preroll + t) % T])
  torch.cuda.synchronize(device)

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize(device)

  # ---- timed region: K steps, per-step events on the env's stream, L2 flushed in between --------
  starts = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
  ends = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
  sampler = ClockSampler(local_rank)
  launches0 = env.launch_count
  probe0 = regime_probe(env)
  barrier()
  sampler.start()
  wall0 = time.perf_counter()
  for k in range(K):
    env._actions.copy_(actions[(W + k) % T])
    flush.zero_()
    stream.wait_stream(torch.cuda.current_stream(device))
    starts[k].record(stream)
    last = env.step(env.actions_buffer)
    ends[k].record(stream)
  barrier()
  wall = time.perf_counter() - wall0
  clocks = sampler.stop()
  if args.dump_outputs and rank == 0:  # before the legs below step the env on
    dump_outputs(args.dump_outputs, *last)
  launches = env.launch_count - launches0
  probe1 = regime_probe(env)
  step_ms = [s.elapsed_time(e) for s, e in zip(starts, ends)]
  total_ms = float(sum(step_ms))
  regime = regime_block(probe0, probe1, K)

  # back-to-back (warm L2, graph launches pipelined) for comparison
  barrier()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record(stream)
  for k in range(K):
    env.step(actions[k % T])
  e1.record(stream)
  barrier()
  warm_ms = e0.elapsed_time(e1)

  # ---- end to end through cr_step_host with pinned host buffers ---------------------------------
  # Per rank: host clock between two stream synchronisations (every step_host ends with one); the
  # ranks are aligned by a barrier BEFORE the window, the max over ranks is taken afterwards.
  h_actions = torch.randint(0, 17, (T, B), dtype=torch.int32).pin_memory()
  h_reward = torch.zeros(B, dtype=torch.float32).pin_memory()
  h_done = torch.zeros(B, dtype=torch.bool).pin_memory()
  for k in range(min(W, 20)):
    env.step_host(h_actions[k % T], h_reward, h_done)
  barrier()
  t0 = time.perf_counter()
  for k in range(K):
    env.step_host(h_actions[k % T], h_reward, h_done)
  e2e_s = time.perf_counter() - t0

  # ---- the same call with the observation batch copied to pinned host memory too (what a host-side
  # learner that consumes pixels pays: B*H*W*3 bytes over PCIe every step); reported beside e2e.
  K_obs, e2e_obs_s = min(K, 200), -1.0
  obs_bytes = B * cfg['size'][0] * cfg['size'][1] * 3
  try:
    h_obs = torch.empty(B, cfg['size'][1], cfg['size'][0], 3, dtype=torch.uint8).pin_memory()
    for k in range(5):
      env.step_host(h_actions[k % T], h_reward, h_done, h_obs)
    barrier()
    t0 = time.perf_counter()
    for k in range(K_obs):
      env.step_host(h_actions[k % T], h_reward, h_done, h_obs)
    e2e_obs_s = time.perf_counter() - t0
  except Exception as exc:  # reported as null; every other number is already measured
    print(f'e2e_obs_to_host skipped: {exc!r}', file=sys.stderr)

  # ---- per-kernel durations inside the step graph (roofline legs), rank 0's batch ------------------
  kt_n, kt = 0, {}
  try:
    kt_n, kt = kernel_times(kwargs, 0, rank * B, env.state_dict(), actions, min(max(K, 100), 400))
  except Exception as exc:
    print(f'kernel_times skipped: {exc!r}', file=sys.stderr)
  # stand-alone launches of the render kernel over the same steady-state batch: cold (L2 flushed) and warm
  R = 30
  def render_alone(cold):
    r0 = [torch.cuda.Event(enable_timing=True) for _ in range(R)]
    r1 = [torch.cuda.Event(enable_timing=True) for _ in range(R)]
    for k in range(R):
      if cold:
        flush.zero_()
      stream.wait_stream(torch.cuda.current_stream(device))
      r0[k].record(stream)
      crafter_b200.env._cabi.check(env._lib.cr_render(env._handle, env._obs.data_ptr(), stream.cuda_stream))
      r1[k].record(stream)
    torch.cuda.synchronize(device)
    return float(sum(a.elapsed_time(b) for a, b in zip(r0, r1)) / R)
  render_cold_ms, render_plain_ms = render_alone(True), render_alone(False)
  # ... and launched the way the step launches it (night frames first, the views k_view prepared in the last
  # step: the state has not changed since)
  os.environ['CRAFTER_B200_RENDER_AS_STEP'] = '1'
  try:
    render_warm_ms = render_alone(False)
  finally:
    os.environ.pop('CRAFTER_B200_RENDER_AS_STEP', None)
  probe2 = regime_probe(env)

  stats = torch.tensor([total_ms, warm_ms, e2e_s * 1e3, e2e_obs_s * 1e3], dtype=torch.float64, device=device)
  if world > 1:
    dist.all_reduce(stats, op=dist.ReduceOp.MAX)
  total_ms, warm_ms, e2e_ms, e2e_obs_ms = stats.tolist()

  if rank == 0:
    peaks_path = ROOT / 'MEASURED_PEAKS.json'
    if peaks_path.exists():
      peak, peak_src = float(json.loads(peaks_path.read_text())['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    else:
      peak, peak_src = 6650.0, 'fallback (B200_PROFILING.md)'
    algo_bytes = render_bytes_per_env(cfg) * B
    # One launch of k_render over the whole batch at the steady-state phase mix is what the roofline is quoted
    # on: every env's frame, warm L2, launched as the step launches it.
    roof_kernel = 'k_render'
    render_ms = render_warm_ms
    achieved = algo_bytes / (render_ms * 1e-3) / 1e9
    traffic, traffic_src, issue = None, None, None
    tpath = ROOT / 'profiles' / 'render_traffic.json'
    if tpath.exists() and args.config == 'default':
      tj = json.loads(tpath.read_text())
      traffic = tj.get('dram_bytes_per_launch')
      traffic_src = tj.get('source', 'profiles/render_traffic.json (last ncu --set full capture of k_render)')
      winst, mhz = tj.get('warp_instructions_per_launch'), clocks.get('sm_mhz')
      if winst and mhz:
        # the bound this kernel actually runs against: warp-instruction issue slots (SMs x 4 schedulers x clock)
        sms = torch.cuda.get_device_properties(device).multi_processor_count
        floor_ms = winst / (sms * 4 * mhz * 1e6) * 1e3
        issue = {'warp_instructions_per_launch': winst, 'issue_floor_ms': floor_ms, 'frac': floor_ms / render_ms,
                 'source': traffic_src, 'note': 'fraction of the issue-slot ceiling at the sampled SM clock'}
    night = float(((probe2[0] % 300 >= 148) & (probe2[0] % 300 <= 272)).float().mean())
    out = {
        'metric': METRIC, 'value': world * B * K / (total_ms * 1e-3), 'unit': UNIT, 'n_gpus': world,
        'steps': K, 'warmup': W, 'ms_per_step': total_ms / K, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'int32/f64', 'data': 'synthetic',
        'config': workload_config(args.config, world, args.preroll),
        'regime': regime,
        'value_warm_l2': world * B * K / (warm_ms * 1e-3), 'ms_per_step_warm_l2': warm_ms / K,
        'clocks': clocks,
        'e2e': {'value': world * B * K / (e2e_ms * 1e-3), 'unit': UNIT, 'h2d_bytes_per_step': 4 * B,
                'd2h_bytes_per_step': 5 * B, 'api': 'Env.step_host -> cr_step_host (pinned host '
                'actions in, reward+done out, stream sync per step); obs stays in HBM',
                'timing': 'host clock per rank between stream synchronisations, max over ranks afterwards'},
        'e2e_obs_to_host': None if e2e_obs_ms <= 0 else {
            'value': world * B * K_obs / (e2e_obs_ms * 1e-3), 'unit': UNIT, 'steps': K_obs,
            'h2d_bytes_per_step': 4 * B, 'd2h_bytes_per_step': 5 * B + obs_bytes,
            'api': 'cr_step_host with obs_host: the observation batch is copied to pinned host memory too '
                   '(PCIe-bound; the north star keeps obs in HBM)'},
        'gpu_launches': launches,
        'roofline': {'kernel': roof_kernel, 'bound': 'hbm', 'achieved': achieved, 'peak': peak,
                     'unit': 'GB/s', 'frac': achieved / peak, 'traffic': traffic, 'traffic_source': traffic_src,
                     'peak_source': peak_src, 'algorithmic_bytes_per_launch': algo_bytes,
                     'ms_per_launch': render_ms,
                     'ms_per_launch_alone_cold_l2': render_cold_ms, 'ms_per_launch_alone_warm_l2': render_warm_ms,
                     'ms_per_launch_alone_warm_l2_env_order_own_gathers': render_plain_ms,
                     'ms_per_launch_in_graph': kt.get('k_render'), 'issue': issue,
                     'night_fraction': night,
                     'how': f'{R} launches of k_render over all {B} envs at the steady-state phase mix, back to back '
                            '(warm L2, night frames first and the views k_view prepared, as inside the step), CUDA '
                            'events on the launch stream',
                     'note': 'not HBM-bound: the obs batch stays in the 126 MB L2 and the reference arithmetic '
                             '(FP64 mix, truncating casts, per-pixel night noise) makes the kernel issue-bound '
                             '(`issue`); inside the step it shares the SMs with world generation (ms_per_launch_in_graph)'},
        'kernels_ms_in_graph': kt, 'kernels_steps': kt_n,
        'wall_s_timed_region': wall,
    }
    if kt.get('k_wg_mat'):
      # worldgen (north star: "render and worldgen kernels"): FP64 simplex terrain, algorithmic bytes
      # per generated world = area bytes of terrain + 256 B of permutation table (SURVEY.md 8d)
      worlds = regime['resets_per_step']
      wg_bytes = (cfg['area'][0] * cfg['area'][1] + 256) * worlds
      out['roofline_worldgen'] = {
          'kernel': 'k_wg_mat', 'bound': 'hbm', 'achieved': wg_bytes / (kt['k_wg_mat'] * 1e-3) / 1e9, 'peak': peak,
          'unit': 'GB/s', 'frac': wg_bytes / (kt['k_wg_mat'] * 1e-3) / 1e9 / peak,
          'algorithmic_bytes_per_launch': wg_bytes, 'worlds_per_launch': worlds, 'ms_per_launch': kt['k_wg_mat'],
          'note': 'FP64-ALU / issue-bound by nature (5-11 OpenSimplex evaluations of ~850 instructions per '
                  'byte of terrain): the HBM fraction is tiny by construction, reported because the north star asks'}
    if not args.no_cpu_baseline and world == 1:
      out['cpu_baseline'] = cpu_baseline(cfg, os.cpu_count() or 1, min(args.preroll, 600))
    print(json.dumps(out))
  if world > 1:
    dist.barrier()
    dist.destroy_process_group()


if __name__ == '__main__':
  main()
