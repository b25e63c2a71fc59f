"""Host-side checks that need no GPU: blob layout, C-ABI surface, loud failure without CUDA."""
import ctypes
import os
import re

import numpy as np
import pytest

from dm_control_b200 import lib as blib
from dm_control_b200 import model as bmodel
from dm_control_b200 import testing_models as tm

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
  assert os.path.exists(blib.SO_PATH), 'build first: python -c "import __graft_entry__ as g; g.build()"'
  L = ctypes.CDLL(blib.SO_PATH)
  header = open(blib.HEADER).read()
  declared = set(re.findall(r'\b(b200mj_\w+)\s*\(', re.sub(r'/\*.*?\*/', '', header, flags=re.S)))
  assert declared == set(blib.SYMBOLS)
  for sym in declared:
    assert hasattr(L, sym), sym
  L.b200mj_version.restype = ctypes.c_char_p
  assert b'b200mj' in L.b200mj_version()
  L.b200mj_error_string.restype = ctypes.c_char_p
  assert L.b200mj_error_string(0) == b'ok'


def test_io_struct_matches_header_order():
  names = [n for n, _ in blib.IO_FIELDS]
  assert names[:5] == ['qpos', 'qvel', 'act', 'qacc_warmstart', 'time']
  assert 'ctrl' in names and 'warning' == names[-1]
  assert ctypes.sizeof(blib.IO) == 8 * len(names)


def test_blob_directory_round_trip():
  m = tm.load('humanoid')
  idata, rdata = m.pack()
  nf = len(bmodel.FIELDS)
  for k, (name, kind) in enumerate(bmodel.FIELDS):
    off, ln = idata[2 * k], idata[2 * k + 1]
    src = m.fields[name].reshape(-1)
    assert ln == src.size, name
    got = idata[off:off + ln] if kind == 'i' else rdata[off:off + ln]
    np.testing.assert_array_equal(got, src, err_msg=name)
  assert idata[0] == 2 * nf   # first field starts right after the directory


def test_model_sizes_match_survey_table():
  # SURVEY.md §8 size table (counted from the reference XML)
  exp = dict(cartpole=dict(nbody=3, njnt=2, nq=2, nv=2, nu=1, na=0, ngeom=5, nsensordata=0),
             cheetah=dict(nbody=8, njnt=9, nq=9, nv=9, nu=6, na=0, ngeom=9, nsensordata=3),
             humanoid=dict(nbody=17, njnt=22, nq=28, nv=27, nu=21, na=0, ngeom=20, nsensordata=66),
             quadruped=dict(nbody=18, njnt=17, nq=23, nv=22, nu=12, na=12, ngeom=20, nsensordata=36, ntendon=12, neq=4),
             cmu_humanoid=dict(nq=63, nv=62, nu=56, na=0, njnt=57, nsensordata=25))
  for name, sizes in exp.items():
    m = tm.load(name)
    for k, v in sizes.items():
      assert getattr(m, k) == v, (name, k, getattr(m, k), v)
  assert abs(tm.load('cheetah').body_mass.sum() - 14.0) < 1e-9          # <compiler settotalmass="14"/>
  assert tm.load('cartpole').opt.integrator == 1                         # RK4 (suite/cartpole.xml:6)
  assert tm.load('humanoid').opt.timestep == 0.005


def test_model_save_load_round_trip(tmp_path):
  m = tm.load('cheetah')
  p = str(tmp_path / 'm.npz')
  m.save(p)
  m2 = bmodel.Model.load(p)
  for f, _ in bmodel.FIELDS:
    np.testing.assert_array_equal(m.fields[f], m2.fields[f])
  assert m2.name2id('bthigh', 'joint') == m.name2id('bthigh', 'joint')
  with pytest.raises(ValueError):
    m2.name2id('nope', 'joint')


def test_no_cpu_fallback():
  import torch
  if torch.cuda.is_available():
    pytest.skip('GPU present')
  from dm_control_b200.physics import BatchedPhysics
  with pytest.raises(blib.EngineError):
    BatchedPhysics(tm.load('cartpole'), batch=2)


def test_model_disable_context_and_errors():
  # dm_control/mujoco/wrapper/core_test.py:291-338 (flag plumbing; the physics effect is tested on the GPU)
  m = tm.load('cartpole').copy()
  base = m.opt.disableflags
  with m.disable('contact', 'gravity'):
    assert m.opt.disableflags == base | (1 << 4) | (1 << 6)
    with m.disable(1 << 10):
      assert m.opt.disableflags & (1 << 10)
  assert m.opt.disableflags == base
  with pytest.raises(ValueError):
    with m.disable('invalid_flag_name'):
      pass
  with pytest.raises(ValueError):
    with m.disable(-99):
      pass


def test_action_spec():
  # dm_control/mujoco/engine_test.py:606-625
  import types
  from dm_control_b200 import mjcf_compile as mc, physics as ph
  xml = '''<mujoco><worldbody><body><geom type="sphere" size="0.1"/><joint type="hinge" name="hinge"/></body></worldbody>
  <actuator><motor joint="hinge" ctrllimited="false"/><motor joint="hinge" ctrllimited="true" ctrlrange="-1 2"/></actuator></mujoco>'''
  lo, hi = ph.action_spec(types.SimpleNamespace(model=mc.compile_xml(xml)))
  np.testing.assert_array_equal(lo, [-1e10, -1.0])
  np.testing.assert_array_equal(hi, [1e10, 2.0])
