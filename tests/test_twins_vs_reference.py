"""The batched torch twins of reference utilities against vectors the REFERENCE'S OWN implementation produced (imported
unmodified through tests/refshim by tools/make_reference_goldens.py) — not against a restatement. The vectors are
stored in tests/golden/reference_twins.npz, so these tests need no reference checkout.

  * dm_control_b200/rewards.py            vs dm_control/utils/rewards.py:25-135            (every sigmoid, bounds, margins)
  * dm_control_b200/control.compute_n_steps vs dm_control/rl/control.py:168-194            (values and error cases)
  * the batched tasks                     vs the task files' own observation / reward code on the same (stored) states
  * BatchedEnvironment's step loop        vs the reference's `control.Environment` across a time limit
(The reference's task files themselves drove the engine for tests/test_reference_tasks.py.)
"""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, 'tests', 'golden', 'reference_twins.npz')

SIGMOIDS = ('gaussian', 'hyperbolic', 'long_tail', 'reciprocal', 'cosine', 'linear', 'quadratic', 'tanh_squared')
TOLERANCE_X = np.concatenate([np.random.RandomState(0).uniform(-6, 6, 400), [-1.0, 0.0, 0.5, 1.0, 2.0, 3.0]])
TOLERANCE_ERROR_CASES = (dict(bounds=(1.0, 0.0)), dict(margin=-1.0), dict(margin=1.0, sigmoid='nope'),
                         dict(margin=1.0, sigmoid='gaussian', value_at_margin=0.0), dict(margin=1.0, sigmoid='linear', value_at_margin=1.0))
N_STEPS_CASES = ((0.025, 0.005), (0.03, 0.005), (0.02, 0.0025), (0.01, 0.01), (0.04, 0.002))
N_STEPS_ERROR_CASES = ((0.005, 0.01), (0.0251, 0.005))
# the batched-task rollouts: seed of the batched environment, batch, random-action steps (actions: RandomState(0))
TWIN_SEED, TWIN_BATCH, TWIN_STEPS = 2, 4, 8
SKIP_KEYS = ('force_torque', 'imu')      # acceleration-stage sensors: after a step they belong to the previous mj_forward
LOOP_TIME_LIMIT, LOOP_STEPS = 0.055, 9   # 5.5 control steps of 0.01 s: the episode ends on the 6th


def tolerance_cases(sigmoid):
  return (((0.0, 0.0), 1.0, 0.1), ((-1.0, 2.0), 0.5, 0.3), ((1.4, float('inf')), 0.35, 0.1),
          ((3.0, 3.0), 3.0, 0.0 if sigmoid in ('cosine', 'linear', 'quadratic') else 0.05), ((0.0, 1.0), 0.0, 0.1))


@pytest.fixture(scope='module')
def ref():
  return np.load(GOLD)


@pytest.mark.parametrize('sigmoid', SIGMOIDS)
def test_tolerance_equals_the_reference(ref, sigmoid):
  from dm_control_b200 import rewards
  np.testing.assert_array_equal(ref['tolerance_x'], TOLERANCE_X)
  for k, (bounds, margin, vam) in enumerate(tolerance_cases(sigmoid)):
    got = rewards.tolerance(torch.as_tensor(TOLERANCE_X), bounds=bounds, margin=margin, sigmoid=sigmoid, value_at_margin=vam).numpy()
    np.testing.assert_allclose(got, ref[f'tolerance_{sigmoid}_{k}'], rtol=1e-13, atol=1e-15)


def test_tolerance_errors_equal_the_reference(ref):
  from dm_control_b200 import rewards
  assert len(ref['tolerance_errors']) == len(TOLERANCE_ERROR_CASES)
  for kw, want in zip(TOLERANCE_ERROR_CASES, ref['tolerance_errors']):
    with pytest.raises(ValueError) as b:
      rewards.tolerance(torch.tensor([0.5], dtype=torch.float64), **kw)
    assert str(b.value) == str(want)


def test_compute_n_steps_equals_the_reference(ref):
  from dm_control_b200 import control
  assert [control.compute_n_steps(ct, pt) for ct, pt in N_STEPS_CASES] == ref['n_steps'].tolist()
  assert len(ref['n_steps_errors']) == len(N_STEPS_ERROR_CASES)
  for (ct, pt), want in zip(N_STEPS_ERROR_CASES, ref['n_steps_errors']):
    with pytest.raises(ValueError) as b:
      control.compute_n_steps(ct, pt)
    assert str(b.value) == str(want)


# ---- the batched task layer (dm_control_b200/suite/*) against the reference's own task files ---------------------------
_TASK_CHILD = r'''
import os, sys, json
sys.path.insert(0, %(root)r); sys.path.insert(0, %(root)r + '/tests'); sys.path.insert(0, %(root)r + '/tests/emu')
import gpu_shim; gpu_shim.install()
import numpy as np, torch
import test_twins_vs_reference as t
from dm_control_b200 import suite as bsuite
dom, task, B, S = %(dom)r, %(task)r, t.TWIN_BATCH, t.TWIN_STEPS
z = np.load(t.GOLD)
tag = 'task_%%s_%%s' %% (dom, task)
keys = [str(k) for k in z[tag + '_keys']]

def load_state(env, qpos, qvel, act, ctrl):
  phys = env.physics
  d = phys.data
  d.qpos.copy_(torch.as_tensor(qpos)); d.qvel.copy_(torch.as_tensor(qvel))
  if phys.model.na:
    d.act.copy_(torch.as_tensor(act))
  phys.set_control(torch.as_tensor(ctrl, device=phys.device))
  phys.forward()
  obs, rew = env.task.get_observation(phys), env.task.get_reward(phys)
  assert set(keys) == set(obs), (keys, sorted(obs))
  return torch.cat([obs[k].reshape(len(qpos), -1) for k in keys if k not in t.SKIP_KEYS], dim=1).cpu().numpy(), rew.cpu().numpy()

worst = {}
# the task code on the stored states (every step of the rollout at once) against the reference's vectors
env = bsuite.load(dom, task, batch=S * B, seed=t.TWIN_SEED, outputs='all')
env.reset()
nu = env.physics.model.nu
g = np.random.RandomState(0)
ctrl = np.stack([g.uniform(-1, 1, (B, nu)) for _ in range(S)])          # the rollout's actions
st = {k: z['state_%%s_%%s' %% (dom, k)].reshape(S * B, -1) for k in ('qpos', 'qvel', 'act')}
obs, rew = load_state(env, st['qpos'], st['qvel'], st['act'], ctrl.reshape(S * B, nu))
worst['observation'] = float(np.abs(obs - z['obs_' + dom].reshape(S * B, -1)).max())
worst['reward'] = float(np.abs(rew - z[tag + '_reward'].reshape(-1)).max())
# the step pipeline: what env.step returns == the task code after a forward() on the state the step left
benv = bsuite.load(dom, task, batch=B, seed=t.TWIN_SEED, outputs='all')
benv.reset()
probe = bsuite.load(dom, task, batch=B, seed=t.TWIN_SEED, outputs='all')
probe.reset()
g = np.random.RandomState(0)
worst['step observation'] = worst['step reward'] = 0.0
for step in range(S):
  a = g.uniform(-1, 1, (B, benv.physics.model.nu))
  ts = benv.step(torch.as_tensor(a, device=benv.physics.device))
  assert set(keys) == set(ts.observation), (keys, sorted(ts.observation))
  got = torch.cat([ts.observation[k].reshape(B, -1) for k in keys if k not in t.SKIP_KEYS], dim=1).cpu().numpy()
  d = benv.physics.data
  want, want_rew = load_state(probe, d.qpos.cpu(), d.qvel.cpu(), d.act.cpu(), a)
  worst['step observation'] = max(worst['step observation'], float(np.abs(got - want).max()))
  worst['step reward'] = max(worst['step reward'], float(np.abs(ts.reward.cpu().numpy() - want_rew).max()))
print('RESULT', json.dumps(worst))
'''


@pytest.mark.timeout(900)
@pytest.mark.parametrize('dom,task', [('cartpole', 'swingup'), ('cheetah', 'run'), ('humanoid', 'run'), ('humanoid', 'stand'), ('quadruped', 'walk')])
def test_batched_tasks_equal_the_reference_task_code(dom, task):
  """Observations and rewards of the batched tasks == what the reference's own `suite/<domain>.py` task computed on the
  same states (stored states of a random-action rollout, so the check does not depend on the physics trajectory); and
  what `env.step` returns == the same task code after a forward() on the state the step left (kernels from the CPU
  emulation build)."""
  import json, subprocess
  r = subprocess.run([sys.executable, '-c', _TASK_CHILD % dict(root=ROOT, dom=dom, task=task)], env=dict(os.environ, B200MJ_EMULATE_GPU='1'),
                     capture_output=True, text=True, timeout=800)
  assert r.returncode == 0, (r.stdout[-1000:], r.stderr[-3000:])
  worst = json.loads(r.stdout.split('RESULT', 1)[1])
  assert len(worst) == 4, worst
  assert max(worst.values()) < 1e-12, worst


_LOOP_CHILD = r'''
import os, sys, json
sys.path.insert(0, %(root)r); sys.path.insert(0, %(root)r + '/tests'); sys.path.insert(0, %(root)r + '/tests/emu')
import gpu_shim; gpu_shim.install()
import torch
import test_twins_vs_reference as t
from dm_control_b200 import suite as bsuite
benv = bsuite.load('cartpole', 'balance', batch=3, seed=0, time_limit=t.LOOP_TIME_LIMIT)
bseq = []
tb = benv.reset(); bseq.append((int(tb.step_type[0]), None))
for _ in range(t.LOOP_STEPS):
  tb = benv.step(torch.zeros(3, 1, dtype=torch.float64, device=benv.physics.device))
  bseq.append((int(tb.step_type[1]), None if tb.discount is None else float(tb.discount[1])))
print('RESULT', json.dumps(bseq))
'''


@pytest.mark.timeout(900)
def test_environment_loop_equals_the_reference_loop(ref):
  """step_type / discount sequence across a time limit and the automatic reset that follows: `BatchedEnvironment`
  (dm_control_b200/control.py) next to the reference's `control.Environment` (rl/control.py:77-127) on cartpole:balance."""
  import json, subprocess
  r = subprocess.run([sys.executable, '-c', _LOOP_CHILD % dict(root=ROOT)], env=dict(os.environ, B200MJ_EMULATE_GPU='1'),
                     capture_output=True, text=True, timeout=800)
  assert r.returncode == 0, (r.stdout[-1000:], r.stderr[-3000:])
  got = [tuple(s) for s in json.loads(r.stdout.split('RESULT', 1)[1])]
  ref = [(int(s), None if np.isnan(d) else float(d)) for s, d in ref['loop_sequence']]     # NaN: no discount (FIRST)
  out = dict(ref=ref, batched=got)
  assert [s for s, _ in ref].count(2) >= 1 and [s for s, _ in ref].count(0) >= 2      # an end and a restart were seen
  # identical up to and including the LAST step (same step count to the time limit, discount 1.0 there) ...
  k = [s for s, _ in ref].index(2)
  assert ref[:k + 1] == got[:k + 1], out
  # ... then the one documented difference of a lock-stepped batch: the reference's next call only resets and returns
  # FIRST (rl/control.py:101-102), the batched environment resets that environment in place AND takes the step (the other
  # environments of the batch cannot wait), so its sequence is the reference's without that FIRST entry
  assert ref[k + 1][0] == 0
  assert ref[k + 2:] == got[k + 1:len(ref) - 1], out
