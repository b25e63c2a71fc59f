"""north_star: "suite tasks run unchanged". The UNMODIFIED reference sources — dm_control/rl/control.py (Environment),
dm_control/suite/{humanoid,cartpole,cheetah,quadruped}.py (tasks + Physics subclasses, incl. the model editing cartpole.py
and quadruped.py do with lxml), suite/base.py, suite/common, suite/utils/randomizers.py, utils/rewards.py,
utils/containers.py, utils/xml_tools.py — drove a B = 1 view of the batched CUDA engine (dm_control_b200/refview.py,
tests/refshim wires the few absent third-party modules): humanoid:run for 100 control steps, the other BASELINE suite
configs and eight further domains for 20 (tools/probe_reference_suite.py sweeps all 47 tasks of the reference suite: 30
run, 17 are refused for a named unsupported feature). tools/make_reference_goldens.py stored, per task, the model the
task file built, the state its `reset` left, and what the run saw step by step, in tests/golden/reference_tasks.npz.

Here the engine is stepped from that state on that model with the same seeded actions, and checked against the CPU
oracle stepped alongside and against the stored contact counts:
  * `-m gpu` twin: runs on the device (or under B200MJ_EMULATE_GPU=1);
  * CPU-collectable test: runs the same body in a child process against the CPU emulation build of the kernels."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, 'tests', 'golden', 'reference_tasks.npz')


def _replay(domain, task):
  """-> (B = 1 view, oracle, stored run, actions) of `domain:task`: view and oracle both start from the state the
  reference's `reset` left; the actions are the run's seeded uniform draws within the action spec."""
  import io
  from dm_control_b200 import refview
  from dm_control_b200.model import Model
  from oracle import oracle as om
  name = f'{domain}_{task}'
  with np.load(GOLD) as z:
    run = {k[len(name) + 1:]: z[k] for k in z.files if k.startswith(name + '/')}
    model = Model.load(io.BytesIO(z['model/' + str(run['model'])].tobytes()))
  phys = refview.SingleEnvPhysics(model)
  start = {k[len('start_'):]: v for k, v in run.items() if k.startswith('start_')}     # absent: zero, as the view starts
  for k, v in start.items():
    np.copyto(phys.data._arrays[k], v)
  o = om.OraclePhysics(model)
  o.qpos[:] = start.get('qpos', 0.0); o.qvel[:] = start.get('qvel', 0.0)
  if model.na:
    o.act[:] = start.get('act', 0.0)
  o.forward()
  (action_seed, nsteps), = [(a, n) for d, t, _, a, n in RUNS if (d, t) == (domain, task)]
  rs = np.random.RandomState(action_seed)
  actions = [rs.uniform(run['action_minimum'], run['action_maximum']) for _ in range(nsteps)]
  return phys, o, run, actions


def run_unmodified_humanoid(nsteps=100):
  phys, o, run, actions = _replay('humanoid', 'run')
  assert o.ncon == 0                                          # humanoid.py:160-166: re-drawn until contact-free
  assert _batched_observation_keys('humanoid', 'run') == [str(k) for k in run['observation_keys']] == sorted(
      ['joint_angles', 'head_height', 'extremities', 'torso_vertical', 'com_velocity', 'velocity'])
  nsub = int(run['n_sub_steps'])
  worst = 0.0
  for t, a in enumerate(actions):
    phys.set_control(a); phys.step(nsub)                      # what control.Environment.step does to the physics
    o.ctrl[:] = a; o.control_step(nsub)
    worst = max(worst, float(np.abs(phys.data.qpos - o.qpos).max()), float(np.abs(phys.data.qvel - o.qvel).max()) * 0.1)
    assert phys.data.ncon == o.ncon == run['ncon'][t]
    assert [(c.geom1, c.geom2) for c in phys.data.contact] == [(c.geom1, c.geom2) for c in o.contact]
    # the reference task's own observation code, on the oracle's numbers
    np.testing.assert_allclose(run['joint_angles'][t], o.qpos[7:], atol=1e-6)
    np.testing.assert_allclose(run['head_height'][t], np.asarray(o.xpos).reshape(-1, 3)[phys.model.name2id('head', 'body'), 2], atol=1e-6)
  assert abs(phys.time() - nsteps * 0.025) < 1e-9
  assert worst < 1e-6, worst
  return worst


def _batched_observation_keys(domain, task):
  """Observation keys of this repo's batched twin of the task."""
  from dm_control_b200 import suite as bsuite
  return sorted(bsuite.load(domain, task, batch=1, seed=0).reset().observation)


def run_unmodified(domain, task, batched=False):
  """Any of the BASELINE suite configs as the reference's own task file ran it: built (the file's own model editing where
  it has any: cartpole.py:104-127, quadruped.py:55-93), reset (its own randomisation), stepped with random actions;
  the engine against the oracle stepped from the same post-reset state. Convex (MPR) contacts end the comparison of an
  episode (DESIGN.md 3: discontinuous in the pose). `batched`: the task has a batched twin here, whose observation
  keys must be the reference task's."""
  phys, o, run, actions = _replay(domain, task)
  nsub = int(run['n_sub_steps'])
  gtype = np.asarray(phys.model.geom_type)
  worst, compared = 0.0, 0
  for t, a in enumerate(actions):
    phys.set_control(a); phys.step(nsub)
    o.ctrl[:] = a; o.control_step(nsub)
    if any(gtype[c.geom1] != 0 and (gtype[c.geom1] > 3 or gtype[c.geom2] > 3) for c in o.contact):
      break
    worst = max(worst, float(np.abs(phys.data.qpos - o.qpos).max()), float(np.abs(phys.data.qvel - o.qvel).max()) * 0.1)
    assert phys.data.ncon == o.ncon == run['ncon'][t]
    assert [(c.geom1, c.geom2) for c in phys.data.contact] == [(c.geom1, c.geom2) for c in o.contact]
    compared += 1
  assert abs(phys.time() - (t + 1) * nsub * phys.timestep()) < 1e-9
  assert compared >= min(10, len(actions)) and worst < 1e-6, (compared, worst)
  out = dict(worst=worst, compared=compared, nsub=nsub)
  if batched:
    out['obs'] = _batched_observation_keys(domain, task)
    assert out['obs'] == [str(k) for k in run['observation_keys']], (out['obs'], run['observation_keys'])
  return out


_SUITE_CASES = [
    ('cartpole', 'swingup', ['position', 'velocity']),                      # BASELINE.json config 0
    ('cartpole', 'balance', ['position', 'velocity']),
    ('cheetah', 'run', ['position', 'velocity']),                           # config 1
    ('quadruped', 'walk', ['egocentric_state', 'force_torque', 'imu', 'torso_upright', 'torso_velocity']),      # config 3
    ('humanoid', 'stand', None), ('humanoid', 'walk', None),
    # domains with no batched twin here: the reference's file + this repo's compiler and engine are all there is
    ('humanoid_CMU', 'stand', None),      # the 62-dof CMU model
    ('acrobot', 'swingup', None), ('fish', 'upright', None), ('hopper', 'hop', None), ('pendulum', 'swingup', None),
    ('point_mass', 'hard', None),         # writes physics.model.wrap_prm in place (point_mass.py:101-112)
    ('reacher', 'hard', None), ('walker', 'run', None), ('cartpole', 'three_poles', None),
]
# the stored runs: (domain, task, the task's random seed, the seed of the uniform actions, control steps)
RUNS = [('humanoid', 'run', 7, 3, 100)] + [(d, t, 5, 11, 20) for d, t, _ in _SUITE_CASES]


@pytest.fixture(scope='module')
def emulated_suite_results():
  """ONE child process (CPU emulation build of the kernels) runs every case; the parametrized tests read their entry."""
  import json
  cases = [(d, t, keys is not None) for d, t, keys in _SUITE_CASES]
  code = ("import os, sys, json, traceback; sys.path.insert(0, %r); sys.path.insert(0, %r); sys.path.insert(0, %r);"
          "import gpu_shim; gpu_shim.install();"
          "import test_reference_tasks as t\n"
          "out = {}\n"
          "for d, k, b in %r:\n"
          "  try: out[d + ':' + k] = t.run_unmodified(d, k, b)\n"
          "  except BaseException as ex: out[d + ':' + k] = dict(error=traceback.format_exc()[-1500:])\n"
          "print('RESULT', json.dumps(out))") % (ROOT, os.path.join(ROOT, 'tests'), os.path.join(ROOT, 'tests', 'emu'), cases)
  env = dict(os.environ, B200MJ_EMULATE_GPU='1')
  r = subprocess.run([sys.executable, '-c', code], env=env, capture_output=True, text=True, timeout=1500)
  assert r.returncode == 0, (r.stdout[-1500:], r.stderr[-3000:])
  return json.loads(r.stdout.split('RESULT', 1)[1])


@pytest.mark.parametrize('domain,task,keys', _SUITE_CASES)
def test_unmodified_reference_suite_tasks_under_emulation(domain, task, keys, emulated_suite_results):
  """The engine on what the reference's own suite/<domain>.py built and drove (CPU emulation build of the kernels, child process)."""
  out = emulated_suite_results[f'{domain}:{task}']
  assert 'error' not in out, out.get('error')
  assert out['compared'] >= 10 and out['worst'] < 1e-6, out
  if keys is not None:
    assert out['obs'] == sorted(keys), out


@pytest.mark.gpu
def test_unmodified_reference_humanoid_task_on_the_engine():
  run_unmodified_humanoid(100)


def test_unmodified_reference_humanoid_task_under_emulation():
  """CPU-collectable twin: the same body in a child process, kernels from the CPU emulation build (tests/emu)."""
  code = ("import os, sys; sys.path.insert(0, %r); sys.path.insert(0, %r); sys.path.insert(0, %r);"
          "import gpu_shim; gpu_shim.install();"
          "import test_reference_tasks as t; print('worst', t.run_unmodified_humanoid(100))") % (
              ROOT, os.path.join(ROOT, 'tests'), os.path.join(ROOT, 'tests', 'emu'))
  env = dict(os.environ, B200MJ_EMULATE_GPU='1')
  r = subprocess.run([sys.executable, '-c', code], env=env, capture_output=True, text=True, timeout=900)
  assert r.returncode == 0, (r.stdout[-1500:], r.stderr[-3000:])
  assert 'worst' in r.stdout
