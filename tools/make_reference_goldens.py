"""Golden vectors from the reference's own PYTHON code (needs a dm_control checkout, see tests/refshim), for machines
that do not have one:

tests/golden/reference_python_vectors.npz, checked by tests/test_reference_goldens.py:

  * `dm_control/utils/rewards.py: tolerance` on a fixed grid for every sigmoid and several (bounds, margin, value_at_margin);
  * the reference task files `dm_control/suite/{cartpole,cheetah,humanoid,quadruped}.py`: `get_observation` / `get_reward`
    evaluated on stored states — the states come from random-action rollouts of this engine (CPU emulation build of the
    kernels), the observation / reward arithmetic is the reference's, run unmodified on the B = 1 reference-facing view.

tests/golden/reference_twins.npz, checked by tests/test_twins_vs_reference.py:
  * `tolerance` on its test grid (values and error messages), `rl/control.py: compute_n_steps` (values and error messages);
  * the task files' observations / rewards on the states of the batched tasks' random-action rollouts (every step),
    and those states (qpos, qvel, act; the controls are the rollout's seeded actions);
  * the `step_type` / `discount` sequence of `control.Environment` across a time limit.

tests/golden/reference_tasks.npz, checked by tests/test_reference_tasks.py: the reference task files run unmodified on the
B = 1 view of the engine; per task the model the file builds (its own MJCF editing, after `reset`), the state `reset`
leaves, its observation keys, and along the seeded random-action rollout the contact counts and (humanoid:run) observations.

Run:  B200MJ_EMULATE_GPU=1 python tools/make_reference_goldens.py
"""
import importlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'tests'), os.path.join(ROOT, 'tests', 'emu')):
  sys.path.insert(0, p)
os.environ['B200MJ_EMULATE_GPU'] = '1'
import gpu_shim; gpu_shim.install()      # noqa: E402,E702
import refshim; refshim.install()        # noqa: E402,E702
import torch                             # noqa: E402
from dm_control_b200 import suite as bsuite      # noqa: E402

SIGMOIDS = ('gaussian', 'hyperbolic', 'long_tail', 'reciprocal', 'cosine', 'linear', 'quadratic', 'tanh_squared')
REWARD_CASES = (((0.0, 0.0), 1.0, 0.1), ((-1.0, 2.0), 0.5, 0.3), ((1.4, float('inf')), 0.35, 0.1), ((0.0, 1.0), 0.0, 0.1))
TASKS = (('cartpole', 'swingup'), ('cartpole', 'balance'), ('cheetah', 'run'), ('humanoid', 'stand'), ('humanoid', 'run'), ('quadruped', 'walk'))
SKIP_KEYS = ('force_torque', 'imu')      # acceleration-stage sensors: not a function of (qpos, qvel, act, ctrl) alone after a step


def main():
  import dm_control.utils.rewards as ref_rewards
  out = {}
  x = np.concatenate([np.linspace(-6, 6, 241), [0.5, 1.4, 1.75, 3.0]])
  out['rewards_x'] = x
  for s in SIGMOIDS:
    for k, (bounds, margin, vam) in enumerate(REWARD_CASES):
      out[f'rewards_{s}_{k}'] = ref_rewards.tolerance(x, bounds=bounds, margin=margin, sigmoid=s, value_at_margin=vam)
  for dom, task in TASKS:
    B = 6
    benv = bsuite.load(dom, task, batch=B, seed=4, outputs='all')
    benv.reset()
    m = benv.physics.model
    g = np.random.RandomState(1)
    mod = importlib.import_module('dm_control.suite.' + dom)
    renv = getattr(mod, task)(random=0)
    renv.reset()
    rphys, rtask = renv.physics, renv.task
    for _ in range(12):      # a short random-action rollout of the batched environment: states off the reset manifold, in contact
      a = g.uniform(-1, 1, (B, m.nu))
      benv.step(torch.as_tensor(a, device=benv.physics.device))
    d = benv.physics.data
    qpos, qvel = d.qpos.cpu().numpy().copy(), d.qvel.cpu().numpy().copy()
    act = d.act.cpu().numpy().copy() if m.na else np.zeros((B, 0))
    obs_rows, rew = [], []
    keys = None
    for e in range(B):
      with rphys.reset_context():
        rphys.data.qpos[:] = qpos[e]; rphys.data.qvel[:] = qvel[e]
        if m.na: rphys.data.act[:] = act[e]
      rphys.set_control(a[e])
      robs = rtask.get_observation(rphys)
      keys = [k for k in robs if k not in SKIP_KEYS]
      obs_rows.append(np.concatenate([np.asarray(robs[k], dtype=np.float64).reshape(-1) for k in keys]))
      rew.append(float(rtask.get_reward(rphys)))
    tag = f'task_{dom}_{task}'
    out[tag + '_qpos'], out[tag + '_qvel'], out[tag + '_act'], out[tag + '_ctrl'] = qpos, qvel, act, a
    out[tag + '_obs'], out[tag + '_reward'] = np.stack(obs_rows), np.array(rew)
    out[tag + '_keys'] = np.array(keys)
    print(tag, 'obs', out[tag + '_obs'].shape, 'reward', np.round(rew, 4))
  path = os.path.join(ROOT, 'tests', 'golden', 'reference_python_vectors.npz')
  np.savez_compressed(path, **out)
  print('wrote', path, os.path.getsize(path), 'bytes')


TWIN_TASKS = (('cartpole', 'swingup'), ('cheetah', 'run'), ('humanoid', 'run'), ('humanoid', 'stand'), ('quadruped', 'walk'))


def _error(fn, *a, **kw):
  try:
    fn(*a, **kw)
  except ValueError as ex:
    return str(ex)
  raise AssertionError(f'{fn.__name__}{a}{kw} did not raise')


def twins():
  import test_twins_vs_reference as t
  import dm_control.utils.rewards as ref_rewards
  import dm_control.rl.control as ref_control
  out = dict(tolerance_x=t.TOLERANCE_X)
  for s in SIGMOIDS:
    for k, (bounds, margin, vam) in enumerate(t.tolerance_cases(s)):
      out[f'tolerance_{s}_{k}'] = ref_rewards.tolerance(t.TOLERANCE_X, bounds=bounds, margin=margin, sigmoid=s, value_at_margin=vam)
  out['tolerance_errors'] = np.array([_error(ref_rewards.tolerance, np.array([0.5]), **kw) for kw in t.TOLERANCE_ERROR_CASES])
  out['n_steps'] = np.array([ref_control.compute_n_steps(ct, pt) for ct, pt in t.N_STEPS_CASES])
  out['n_steps_errors'] = np.array([_error(ref_control.compute_n_steps, ct, pt) for ct, pt in t.N_STEPS_ERROR_CASES])
  for dom, task in TWIN_TASKS:
    B = t.TWIN_BATCH
    benv = bsuite.load(dom, task, batch=B, seed=t.TWIN_SEED, outputs='all')
    benv.reset()
    nu = benv.physics.model.nu
    g = np.random.RandomState(0)
    renv = getattr(importlib.import_module('dm_control.suite.' + dom), task)(random=0)
    renv.reset()
    rphys, rtask = renv.physics, renv.task
    obs, rew, states = [], [], dict(qpos=[], qvel=[], act=[])
    for _ in range(t.TWIN_STEPS):
      a = g.uniform(-1, 1, (B, nu))
      benv.step(torch.as_tensor(a, device=benv.physics.device))
      d = benv.physics.data
      for k in ('qpos', 'qvel', 'act'):
        states[k].append(getattr(d, k).cpu().numpy().copy())
      for e in range(B):
        with rphys.reset_context():
          rphys.data.qpos[:] = d.qpos[e].cpu().numpy(); rphys.data.qvel[:] = d.qvel[e].cpu().numpy()
          if benv.physics.model.na: rphys.data.act[:] = d.act[e].cpu().numpy()
        rphys.set_control(a[e])
        robs = rtask.get_observation(rphys)
        keys = sorted(robs)
        obs.append(np.concatenate([np.asarray(robs[k], dtype=np.float64).reshape(-1) for k in keys if k not in SKIP_KEYS]))
        rew.append(float(rtask.get_reward(rphys)))
    tag = f'task_{dom}_{task}'
    out[tag + '_keys'] = np.array(keys)
    out[tag + '_reward'] = np.array(rew).reshape(t.TWIN_STEPS, B)
    # the states the reference code saw (the controls are the seeded actions) and its observations there: tasks of one
    # domain roll out the same states (same seed, model and actions) and observe them alike, so they are stored once
    per_domain = {f'state_{dom}_{k}': np.stack(v) for k, v in states.items()}
    per_domain[f'obs_{dom}'] = np.stack(obs).reshape(t.TWIN_STEPS, B, -1)
    for k, v in per_domain.items():
      assert k not in out or np.array_equal(out[k], v), (dom, task, k)
      out[k] = v
    print(tag, out[f'obs_{dom}'].shape)
  import dm_control.suite.cartpole as ref_cartpole
  renv = ref_cartpole.balance(time_limit=t.LOOP_TIME_LIMIT, random=0)
  ts = renv.reset()
  seq = [(int(ts.step_type), np.nan)]
  for _ in range(t.LOOP_STEPS):
    ts = renv.step(np.zeros(1))
    seq.append((int(ts.step_type), np.nan if ts.discount is None else float(ts.discount)))
  out['loop_sequence'] = np.array(seq)
  path = os.path.join(ROOT, 'tests', 'golden', 'reference_twins.npz')
  np.savez_compressed(path, **out)
  print('wrote', path, os.path.getsize(path), 'bytes')


def task_runs():
  """The reference task files through `control.Environment` on the B = 1 view: what tests/test_reference_tasks.py steps
  the engine and the oracle from. One file; a model several tasks share (humanoid.xml, cartpole.xml) is stored once,
  as the bytes of its uncompressed `Model.save` archive so that the file's compression sees all of it."""
  import hashlib
  import io
  import test_reference_tasks as t
  from dm_control_b200 import refview
  out, models = {}, {}
  for domain, task, seed, action_seed, nsteps in t.RUNS:
    name = f'{domain}_{task}'
    env = getattr(importlib.import_module('dm_control.suite.' + domain), task)(random=seed)
    spec = env.action_spec()
    ts = env.reset()
    phys = env.physics
    arrays = phys.data._arrays
    # the view starts zeroed: only the non-zero parts of the state `reset` left are stored
    run = {'start_' + k: np.array(arrays[k]) for k in refview._STATE if k in arrays and k != 'ctrl' and np.any(arrays[k])}
    run['n_sub_steps'] = np.array(int(round(env.control_timestep() / phys.timestep())))
    run['action_minimum'], run['action_maximum'] = np.broadcast_to(spec.minimum, spec.shape), np.broadcast_to(spec.maximum, spec.shape)
    rs = np.random.RandomState(action_seed)
    rows = dict(ncon=[], joint_angles=[], head_height=[])
    for _ in range(nsteps):
      ts = env.step(rs.uniform(spec.minimum, spec.maximum))      # the actions tests/test_reference_tasks.py draws
      rows['ncon'].append(phys.data.ncon)
      if (domain, task) == ('humanoid', 'run'):
        rows['joint_angles'].append(np.array(ts.observation['joint_angles'])); rows['head_height'].append(np.array(ts.observation['head_height']))
    run.update({k: np.array(v, dtype=np.float64) for k, v in rows.items() if v})
    run['observation_keys'] = np.array(sorted(ts.observation))
    saved = io.BytesIO()
    phys._b.model.save(saved)
    plain = io.BytesIO()
    np.savez(plain, **dict(np.load(io.BytesIO(saved.getvalue()))))
    raw = plain.getvalue()
    key = models.setdefault(hashlib.sha1(raw).hexdigest(), name)
    if key == name:
      out[f'model/{name}'] = np.frombuffer(raw, np.uint8)
    run['model'] = np.array(key)
    out.update({f'{name}/{k}': v for k, v in run.items()})
    print(name, 'steps', nsteps, 'nsub', int(run['n_sub_steps']), 'model', key)
  path = os.path.join(ROOT, 'tests', 'golden', 'reference_tasks.npz')
  np.savez_compressed(path, **out)
  print('wrote', path, os.path.getsize(path), 'bytes')


if __name__ == '__main__':
  main()
  twins()
  task_runs()
