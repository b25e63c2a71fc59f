"""bench.py — env-steps/s of suite.humanoid:run, batch 8192 per GPU, random-action rollout (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one rank per GPU under torchrun)
    python bench.py --impl reference --steps K --warmup W    # the CPU restatement of the reference path, host cores
    python bench.py --steps K --dump-outputs DIR             # + the last timed step's TimeStep as DIR/<name>.npy

One "step" = one `Environment.step` for the whole batch = n_sub_steps(5) physics steps + reward + observation
(reference: rl/control.py:99-127, suite/humanoid.py:30). Prints ONE JSON line on rank 0. See DESIGN.md §Measurement.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the tree may be read-only: the benchmark leaves it as it found it

METRIC = 'env-steps/sec suite.humanoid:run batch 8192 (per GPU) random-action rollout'
UNIT = 'env-steps/s'
BATCH = 8192
NSUB = 5
# SURVEY.md §8d: compulsory fp64 bytes per humanoid env-step (5 fused substeps + observation-contract outputs)
ALGO_BYTES_PER_ENV_STEP = 4068
OBS_DIM = 67


def _peaks():
  p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(p):
    return float(json.load(open(p))['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
  return 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler:
  """SM clock + clocks-event (throttle) reasons sampled DURING the timed region.

  Samples are taken inline from the benchmark thread through NVML every few steps (0.15 ms per sample). A polling
  child process (`nvidia-smi -lms 200`) or a polling thread was measured to cost this workload 15-40 %: the step
  issues ~17 launches plus cross-stream events, and concurrent driver queries stall them. nvidia-smi is the fallback
  (one query per sample) when pynvml is unavailable.
  """
  BITS = dict(sw_power_cap=0x4, hw_slowdown=0x8, sw_thermal_slowdown=0x20, hw_thermal_slowdown=0x40)

  def __init__(self, index, uuid=None):
    self.index, self.rows, self.mode = index, [], None
    try:
      import pynvml
      pynvml.nvmlInit()
      h = None
      if uuid:
        for cand in (f'GPU-{uuid}', str(uuid)):
          try:
            h = pynvml.nvmlDeviceGetHandleByUUID(cand.encode())
            break
          except Exception:
            h = None
      self._h = h if h is not None else pynvml.nvmlDeviceGetHandleByIndex(index)
      self._nv = pynvml
      self._max = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
      self._reasons = getattr(pynvml, 'nvmlDeviceGetCurrentClocksEventReasons', None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
      self.mode = 'nvml-inline'
    except Exception:
      self.mode = 'nvidia-smi-inline'

  def sample(self):
    try:
      if self.mode == 'nvml-inline':
        sm = self._nv.nvmlDeviceGetClockInfo(self._h, self._nv.NVML_CLOCK_SM)
        bits = int(self._reasons(self._h))
        self.rows.append((float(sm), float(self._max), [n for n, b in self.BITS.items() if bits & b]))
      else:
        out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=clocks.sm,clocks.max.sm,'
                              'clocks_event_reasons.sw_power_cap,clocks_event_reasons.hw_slowdown,'
                              'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.hw_thermal_slowdown',
                              '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=10).stdout
        f = [x.strip() for x in out.strip().split(',')]
        self.rows.append((float(f[0]), float(f[1]), [n for n, v in zip(self.BITS, f[2:6]) if v.lower().startswith('active')]))
    except Exception:
      pass

  def summary(self):
    sm = [r[0] for r in self.rows]
    return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=max((r[1] for r in self.rows), default=None),
                reasons=sorted({n for r in self.rows for n in r[2]}), samples=len(sm), source=self.mode)


# ------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference path on the host cores
# ------------------------------------------------------------------------------------------------------------
def physical_cores():
  """One logical CPU per physical core (sysfs topology), restricted to this process's affinity mask."""
  allowed = sorted(os.sched_getaffinity(0))
  seen = {}
  for c in allowed:
    try:
      core = open(f'/sys/devices/system/cpu/cpu{c}/topology/core_id').read().strip()
      pkg = open(f'/sys/devices/system/cpu/cpu{c}/topology/physical_package_id').read().strip()
    except OSError:
      core, pkg = str(c), '0'
    seen.setdefault((pkg, core), c)
  return sorted(seen.values())


def _cpu_worker(args):
  """One host process pinned to one physical core: builds its environments, settles them, then rolls out `reps`
  timed windows of `timed_steps` env-steps each inside one C call per environment; every window starts at a barrier."""
  t, cpu, nenv, warmup_steps, timed_steps, reps, barrier = args
  try:
    os.sched_setaffinity(0, {cpu})
  except OSError:
    pass
  import numpy as np
  from dm_control_b200 import testing_models as tm
  from oracle import oracle as om
  model = tm.load('humanoid')
  q0, v0 = tm.initial_states(model, 'humanoid', nenv, 7000 + t)
  envs = []
  for e in range(nenv):
    o = om.OraclePhysics(model)
    o.qpos[:] = q0[e]; o.qvel[:] = v0[e]; o.forward()
    envs.append(o)
  total = warmup_steps + reps * timed_steps
  tape = np.random.RandomState(100 + t).uniform(-1, 1, (total, nenv, model.nu))
  for j, o in enumerate(envs):
    o.rollout(tape[:warmup_steps, j], NSUB)
  spans = []
  for r in range(reps):
    lo = warmup_steps + r * timed_steps
    if barrier is not None:
      barrier.wait()
    t0 = time.time()
    for j, o in enumerate(envs):
      o.rollout(tape[lo:lo + timed_steps, j], NSUB)
    spans.append((t0, time.time()))
  return spans


def _run_cpu(cores, nenv, warm, timed, reps):
  import multiprocessing as mp
  ctx = mp.get_context('fork')
  if len(cores) == 1:
    return [_cpu_worker((0, cores[0], nenv, warm, timed, reps, None))]
  barrier = ctx.Barrier(len(cores))
  procs, pipes = [], []
  def child(conn, a):
    conn.send(_cpu_worker(a)); conn.close()
  for t, cpu in enumerate(cores):
    rx, tx = ctx.Pipe(duplex=False)
    p = ctx.Process(target=child, args=(tx, (t, cpu, nenv, warm, timed, reps, barrier)))
    p.start(); procs.append(p); pipes.append(rx)
  out = [rx.recv() for rx in pipes]
  for p in procs:
    p.join()
  return out


def time_cpu(total_envs=BATCH, warmup_steps=21, reps=3, target_s=3.0):
  """Times `control_step(5)` (legacy ordering, engine.py:147-162) of the scalar CPU oracle on the host's PHYSICAL cores.

  1. calibration: one pinned process alone -> microseconds per physics step per core;
  2. one pinned process per physical core, the BATCH environments split evenly (capped so that a window stays near
     `target_s` seconds of work per process), `reps` timed windows, each started at a barrier; a window's time is the
     span from the first start to the last finish; the best window is reported.
  The window is sized here, not by --steps: the scalar host path would need minutes for --steps x 8192 environments.
  Returns a dict (value = env-steps/s of the best window, steps = env-steps each timed window ran)."""
  from oracle import oracle as om
  om.build()
  cores = physical_cores()
  cal_env, cal_steps = 16, 30
  sp = _run_cpu(cores[:1], cal_env, 5, cal_steps, 1)[0][0]
  us_per_phys = (sp[1] - sp[0]) / (cal_env * cal_steps * NSUB) * 1e6
  nenv = -(-total_envs // len(cores))
  per_env_step_s = us_per_phys * NSUB * 1e-6
  timed = int(max(20, min(400, round(target_s / (nenv * per_env_step_s)))))
  if nenv * timed * per_env_step_s > 2.5 * target_s:        # few cores: bound the window instead of the env count's share
    nenv = max(8, int(2.5 * target_s / (timed * per_env_step_s)))
  spans = _run_cpu(cores, nenv, warmup_steps, timed, reps)
  rates = []
  for r in range(reps):
    dt = max(s[r][1] for s in spans) - min(s[r][0] for s in spans)
    rates.append(nenv * len(cores) * timed / dt)
  best = max(rates)
  single = 1e6 / (us_per_phys * NSUB)                          # env-steps/s of one core alone
  return dict(value=best, unit=UNIT, cores=len(cores), kind='port', steps=timed,
              sample=(f'{nenv * len(cores)} envs ({nenv}/process x {len(cores)} processes, one pinned per physical core) x {timed} '
                      f'env-steps x {reps} windows (best) after {warmup_steps} settle steps, seeded humanoid:run states, uniform(-1,1) actions'),
              per_core_us_per_physics_step=us_per_phys, parallel_efficiency=best / (single * len(cores)),
              windows_env_steps_per_s=rates, work_s_per_process=nenv * timed * per_env_step_s,
              same_config=bool(nenv * len(cores) == total_envs), ms_per_env_step_batch=1e3 * nenv * len(cores) / best)


def run_reference(args):
  rank = int(os.environ.get('RANK', '0'))
  if rank != 0:
    return
  kind, note = 'port', 'restated CPU oracle (oracle/mjoracle.cpp), NOT libmujoco: MuJoCo is absent from this image'
  cpu = None
  try:
    sys.path.insert(0, os.path.join(ROOT, 'tools'))
    import time_mujoco_cpu
    if time_mujoco_cpu.available():      # a machine that has the real reference: time that instead
      ref_steps = max(20, min(args.steps, 300))
      value, cores, sample, ms = time_mujoco_cpu.time_reference(21, ref_steps, 8)
      cpu = dict(value=value, unit=UNIT, cores=cores, kind='reference', steps=ref_steps, sample=sample, ms_per_env_step_batch=ms)
      kind, note = 'reference', 'unmodified dm_control suite.load(humanoid, run) on mujoco, Environment.step'
  except Exception as ex:
    sys.stderr.write(f'real-reference arm failed ({ex!r}); timing the oracle port\n')
    cpu = None
  if cpu is None:
    cpu = time_cpu()
  value = cpu['value']
  line = dict(impl='reference', metric=METRIC, value=value, unit=UNIT, n_gpus=args.gpus, steps=cpu['steps'], warmup=args.warmup,
              ms_per_step=cpu.pop('ms_per_env_step_batch'), higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f64',
              data='synthetic',
              config=dict(workload='suite.humanoid:run', batch_per_gpu=BATCH, n_sub_steps=NSUB, note=note),
              cpu_baseline=cpu, e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
  print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------------
def _mean_ncon(d):
  return float(d.ncon.double().mean()) if hasattr(d, 'ncon') else None


def _time_env(env, steps, warmup, gen_seed, nu, dev):
  """Device-resident env-steps/s of one BatchedEnvironment through env.step (used for the other BASELINE configs)."""
  import torch
  B = env.physics.batch
  gen = torch.Generator(device=dev).manual_seed(gen_seed)
  act = torch.empty(B, nu, dtype=torch.float64, device=dev)
  env.physics.check_errors = False
  if hasattr(env, '_graph_step') and not os.environ.get('B200_BENCH_NO_GRAPH'):
    env._graph_step = True             # one CUDA graph per control step: these small models are launch-bound otherwise
  env.reset()
  env.physics.data.warning.zero_()     # reset procedures embed / re-draw on purpose (quadruped.py:266-270): count the rollout only
  for _ in range(warmup):
    act.uniform_(-1, 1, generator=gen); env.step(act)
  torch.cuda.synchronize(dev)
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for _ in range(steps):
    act.uniform_(-1, 1, generator=gen); env.step(act)
  e1.record(); torch.cuda.synchronize(dev)
  ms = e0.elapsed_time(e1) / steps
  d = env.physics.data
  return dict(batch=B, n_sub_steps=env.n_sub_steps, steps=steps, ms_per_step=ms, env_steps_per_s=B / ms * 1e3,
              physics_steps_per_s=B * env.n_sub_steps / ms * 1e3, mean_ncon=_mean_ncon(d),
              warnings=[int(x) for x in d.warning.sum(0).tolist()])


def _contact_load(snaps, caps):
  import torch
  ncon = torch.cat([s[0] for s in snaps]).double(); nefc = torch.cat([s[1] for s in snaps]).double()
  niter = torch.cat([s[2] for s in snaps]).double()
  pops, lo = [], -1
  for c in caps:
    pops.append(float(((nefc > lo) & (nefc <= c)).double().mean())); lo = c
  return dict(mean_ncon=float(ncon.mean()), mean_nefc=float(nefc.mean()), p99_nefc=float(torch.quantile(nefc, 0.99)),
              max_nefc=float(nefc.max()), mean_niter=float(niter.mean()), bucket_caps=list(caps), bucket_populations=pops,
              note='state after each sampled env-step: ncon / nefc of the trailing mj_step1, solver iterations of its last physics step')


def dump_outputs(out_dir, ts):
  """The TimeStep of the last timed env.step as DIR/<name>.npy (float64): step_type, reward, discount and one file per
  observation (observation.<key>). For batch 8192 that is ~4.6 MB, so nothing is sampled."""
  import numpy as np
  import torch
  os.makedirs(out_dir, exist_ok=True)
  arrays = dict(step_type=ts.step_type, reward=ts.reward, discount=ts.discount)
  arrays.update({f'observation.{k}': v for k, v in ts.observation.items()})
  for name, t in arrays.items():
    np.save(os.path.join(out_dir, name + '.npy'), t.detach().to('cpu', dtype=torch.float64).numpy())


def run_gpu(args):
  import torch
  import torch.distributed as dist
  from dm_control_b200 import lib as blib
  from dm_control_b200 import suite

  world = int(os.environ.get('WORLD_SIZE', '1'))
  rank = int(os.environ.get('RANK', '0'))
  local = int(os.environ.get('LOCAL_RANK', '0'))
  torch.cuda.set_device(local)
  dev = torch.device('cuda', local)
  if world > 1:
    dist.init_process_group('nccl', device_id=dev)
  L = blib.load()

  from dm_control_b200 import sharding
  flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=dev)   # > 126 MB L2

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  def build(batch, seed):
    env = suite.load('humanoid', 'run', batch=batch, seed=seed, device=dev)
    env.physics.check_errors = False   # no device->host sync inside the rollout; warnings are summed at the end
    # the task's ~80 tiny reward/observation launches replay as one CUDA graph (falls back to eager if capture fails)
    env._graph_task_ops = not os.environ.get('B200_BENCH_NO_GRAPH')
    # ... and, where no events are recorded inside the step (the e2e arm), the whole control step as ONE graph
    env._graph_step = not os.environ.get('B200_BENCH_NO_GRAPH')
    # start states: the task's own initialize_episode (suite/humanoid.py:152-166: random joint configuration, rejected
    # until contact-free), then the settle below
    env.reset()
    if os.environ.get('B200_BENCH_START') == 'seeded':
      # round-1 protocol (A/B continuity only): seeded tumbling starts instead of the task's initialize_episode
      from dm_control_b200 import testing_models as tm
      q0, v0 = tm.initial_states(env.physics.model, 'humanoid', batch, seed=rank)
      env.physics.data.qpos.copy_(torch.as_tensor(q0, device=dev)); env.physics.data.qvel.copy_(torch.as_tensor(v0, device=dev))
      env.physics.forward()
    return env

  def runner(env, batch, gather_world):
    model = env.physics.model
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    actions = torch.empty(batch, model.nu, dtype=torch.float64, device=dev)
    packed = torch.empty(batch, OBS_DIM + 2, dtype=torch.float64, device=dev)
    gathered = sharding.alloc_gather(packed, gather_world) if gather_world > 1 else None

    def pack_block(reward, o, discount):
      # device-side epilogue of the control step (captured with it): the observation dict as one [B, 69] block
      packed[:, :21] = o['joint_angles']; packed[:, 21] = o['head_height']; packed[:, 22:34] = o['extremities']
      packed[:, 34:37] = o['torso_vertical']; packed[:, 37:40] = o['com_velocity']; packed[:, 40:67] = o['velocity']
      packed[:, 67] = reward; packed[:, 68] = discount
    env.post_step_hook = pack_block

    def pack(ts):
      if gather_world > 1:
        # NCCL over NVLink: observations/rewards of every rank, in environment order (north_star)
        sharding.gather_packed(packed, gathered)

    def one_step(timing=None):
      flush.fill_(0.0)                                   # L2 flush between timed iterations (inside the timed region)
      actions.uniform_(-1, 1, generator=gen)
      pack(env.step(actions, timing=timing))
    return model, actions, packed, gathered, pack, one_step

  env = build(BATCH, 1000 + rank)
  phys = env.physics
  model, actions, packed, gathered, pack, one_step = runner(env, BATCH, world)

  sampler = ClockSampler(local, getattr(torch.cuda.get_device_properties(local), "uuid", None)) if (rank == 0 and not os.environ.get("B200_BENCH_NO_SAMPLER")) else None
  # settle to the contact load the metric is quoted on (SURVEY §8d: 20 warm-up env-steps minimum)
  try:
    one_step()
  except Exception as ex:           # graph capture unsupported for some op: eager task ops
    if not env._graph_task_ops:
      raise
    sys.stderr.write(f'task-op graph capture failed ({ex!r}); running the task ops eagerly\n')
    env._graph_task_ops = False; env._graph = None
    torch.cuda.synchronize()
    one_step()
  settle = int(os.environ.get('B200_BENCH_SETTLE', max(args.warmup, 20)))     # profiling runs shorten it
  for _ in range(settle):
    one_step()
  barrier()

  # ---- kernel-group time for the roofline: a few eager steps with CUDA events around the one b200mj_step call ------
  nk = min(8, args.steps)
  kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(nk)]
  launches0 = L.b200mj_launch_count()
  for i in range(nk):
    one_step(timing=kev[i])
  torch.cuda.synchronize()
  launches_per_step = (L.b200mj_launch_count() - launches0) / nk
  kernel_ms = sum(a.elapsed_time(b) for a, b in kev) / nk
  one_step(); one_step()                               # back on the graph path (re-captures nothing: same flags)

  # ---- device-resident arm: the user-facing env.step (one CUDA graph per step), inputs generated on the device ----
  ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
  snaps = []
  barrier()
  ev[0].record()
  every = max(1, args.steps // 8)
  for i in range(args.steps):
    if sampler and i % every == every // 2:
      sampler.sample()                                 # clocks / throttle reasons while the region is running
    one_step()
    if i % every == 0:
      snaps.append(tuple(getattr(phys.data, f).clone() if hasattr(phys.data, f) else torch.zeros(BATCH, dtype=torch.int32, device=dev)
                         for f in ('ncon', 'nefc', 'solver_niter')))
  ev[1].record()
  barrier()
  ms_total = ev[0].elapsed_time(ev[1])
  launches = int(round(launches_per_step * args.steps))
  clocks = sampler.summary() if sampler else None
  t = torch.tensor([ms_total, kernel_ms], dtype=torch.float64, device=dev)
  if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
  ms_total, kernel_ms = float(t[0]), float(t[1])
  value = BATCH * world * args.steps / (ms_total * 1e-3)
  desc = phys.describe()
  load = _contact_load(snaps, [b['rows'] for b in desc.get('acc_buckets', [])] or [10, 24, model.njmax])

  # ---- end-to-end arm: HOST action buffer in, HOST observation/reward buffer out, every step -----------------
  # host action tape, drawn before the clock starts (drawing 172k doubles on one host core costs ~0.4 ms per step and
  # is the synthetic policy's time, not the path's); 16 pinned blocks, cycled
  def e2e(env, batch, actions, packed, gathered, pack, gather_world, steps):
    cpu_gen = torch.Generator().manual_seed(77 + rank)
    act_tape = [torch.empty(batch, model.nu, dtype=torch.float64).uniform_(-1, 1, generator=cpu_gen).pin_memory() for _ in range(16)]
    # every rank reads back its own rows of the gathered block over its own PCIe link into pinned host memory
    out_host = torch.empty(batch, OBS_DIM + 2, dtype=torch.float64).pin_memory()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    ts = None
    for i in range(steps):
      flush.fill_(0.0)
      actions.copy_(act_tape[i % len(act_tape)], non_blocking=True)     # H2D from pinned host memory
      ts = env.step(actions)
      pack(ts)
      out_host.copy_(packed, non_blocking=True)                         # D2H of this rank's rows
      torch.cuda.current_stream().synchronize()                         # the user reads obs before the next action
    e1.record()
    barrier()
    tt = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
      dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    return batch * world * steps / (float(tt[0]) * 1e-3), ts

  e2e_value, last_ts = e2e(env, BATCH, actions, packed, gathered, pack, world, args.steps)
  if args.dump_outputs and rank == 0:
    dump_outputs(args.dump_outputs, last_ts)
  warn = phys.data.warning.sum(0)
  if world > 1:
    dist.all_reduce(warn)

  # ---- strong scaling: BASELINE.json "batch 8192, 8xB200 sharded" = the SAME 8192 environments split over N GPUs -----
  strong = None
  if world > 1:
    sb = BATCH // world
    env_s = build(sb, 5000 + rank)
    _, actions_s, packed_s, gathered_s, pack_s, one_step_s = runner(env_s, sb, world)
    for _ in range(settle + 1):
      one_step_s()
    barrier()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    for _ in range(args.steps):
      one_step_s()
    s1.record(); barrier()
    tt = torch.tensor([s0.elapsed_time(s1)], dtype=torch.float64, device=dev)
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    strong = dict(global_batch=BATCH, batch_per_gpu=sb, value=BATCH * args.steps / (float(tt[0]) * 1e-3), unit=UNIT,
                  ms_per_step=float(tt[0]) / args.steps,
                  e2e=e2e(env_s, sb, actions_s, packed_s, gathered_s, pack_s, world, args.steps)[0])

  # ---- the other BASELINE.json configs on one GPU, same run (device-resident, through env.step) ---------------
  configs = None
  if world == 1 and not args.no_configs:
    configs = {}
    for dom, task, B in (('cheetah', 'run', 4096), ('quadruped', 'walk', 4096), ('cartpole', 'swingup', 4096)):
      try:
        e = suite.load(dom, task, batch=B, seed=3, device=dev)
        configs[f'suite.{dom}:{task}'] = _time_env(e, args.steps, 10, 5, e.physics.model.nu, dev)
        e.physics.free()
      except Exception as ex:
        configs[f'suite.{dom}:{task}'] = dict(error=repr(ex))
    try:
      from dm_control_b200 import locomotion
      e = locomotion.load('cmu_humanoid_run_walls', batch=2048, seed=3, device=dev)
      configs['locomotion.cmu_humanoid run-through-corridor (walls)'] = _time_env(e, args.steps, 10, 5, e.physics.model.nu, dev)
      e.physics.free()
      # the same with the walker's 64 x 64 egocentric camera observable, ray-cast on the device every control step (b200mj_render)
      e = locomotion.load('cmu_humanoid_run_walls', batch=2048, seed=3, device=dev, egocentric_camera=True)
      r = _time_env(e, args.steps, 10, 5, e.physics.model.nu, dev)
      r['observation'] = 'walker/egocentric_camera [2048, 64, 64, 3] uint8 per step (ray-cast hand-off, not MuJoCo GL pixels)'
      configs['locomotion.cmu_humanoid run-through-corridor (walls) + egocentric camera'] = r
      e.physics.free()
    except Exception as ex:
      configs['locomotion.cmu_humanoid run-through-corridor (walls)' + (' + egocentric camera' if 'locomotion.cmu_humanoid run-through-corridor (walls)' in configs else '')] = dict(error=repr(ex))

  if rank == 0:
    peak, peak_src = _peaks()
    achieved = ALGO_BYTES_PER_ENV_STEP * BATCH / (kernel_ms * 1e-3) / 1e9
    prof = {}
    pj = os.path.join(ROOT, 'profiles', 'summary.json')
    if os.path.exists(pj):
      prof = json.load(open(pj))
    cpu = None
    if world == 1 and not args.no_cpu:
      cpu = time_cpu()
      cpu.pop('ms_per_env_step_batch', None)
    line = dict(
        metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
        ms_per_step=ms_total / args.steps, higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f64',
        data='synthetic',
        config=dict(workload='suite.humanoid:run', batch_per_gpu=BATCH, global_batch=BATCH * world, n_sub_steps=NSUB,
                    physics_steps_per_s=value * NSUB, parallelism=f'env-sharded x{world}',
                    start_states=f'task.initialize_episode (suite/humanoid.py:152-166) + {settle + 1} settle env-steps',
                    call='BatchedEnvironment.step with graph_step=True: the control step (physics launches on the engine streams + task ops) replayed as one CUDA graph, value and e2e; roofline.kernel_ms from 8 eager steps with CUDA events around the b200mj_step call',
                    actions='uniform(-1,1) generated on device', l2='256 MB flush write between steps, inside the timed region',
                    task_ops='one CUDA-graph replay' if env._graph_task_ops else 'eager torch ops',
                    obs_gather='NCCL all_gather_into_tensor of [B,69] f64 each step; every rank copies its own rows to pinned host memory' if world > 1 else 'n/a (1 GPU)',
                    kernels=desc, nconmax=model.nconmax, njmax=model.njmax),
        e2e=dict(value=e2e_value, unit=UNIT, h2d_bytes_per_step=BATCH * model.nu * 8 * world,
                 d2h_bytes_per_step=BATCH * (OBS_DIM + 2) * 8 * world),
        gpu_launches=int(launches), contact_load=load,
        roofline=dict(bound='hbm', achieved=achieved, peak=peak, unit='GB/s', frac=achieved / peak,
                      traffic=prof.get('dram_bytes_per_step', prof.get('dram_bytes_per_launch')), peak_source=peak_src,
                      kernel='b200mj step group: [pos_kernel, acc_tn_kernel x row-buckets] x n_sub_steps (first pos reused from the previous trailing mj_step1), posfinal_kernel',
                      dominant_kernel=prof.get('dominant_kernel', 'b200mj_acc_tn_kernel'),
                      dominant_kernel_utilisation_pct=prof.get('dominant_kernel_utilisation_pct'),
                      kernel_ms=kernel_ms, kernel_share_of_step=kernel_ms / (ms_total / args.steps),
                      algorithmic_bytes_per_launch=ALGO_BYTES_PER_ENV_STEP * BATCH,
                      note='latency/issue-bound fp64 kernel: compulsory traffic is ~4 kB per env-step, see DESIGN.md'),
        clocks=clocks, warnings=[int(x) for x in warn.tolist()])
    if strong is not None:
      line['strong'] = strong
    if configs is not None:
      line['configs'] = configs
    if cpu is not None:
      line['cpu_baseline'] = cpu
    print(json.dumps(line))
  if world > 1:
    dist.destroy_process_group()


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=200)      # 0.8 s per timed window: a 2 ms hiccup of the shared box is 0.25 %, not 1 %
  ap.add_argument('--warmup', type=int, default=20)
  ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
  ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
  ap.add_argument('--no-configs', action='store_true', help='skip the other BASELINE.json configs (N=1 only)')
  ap.add_argument('--dump-outputs', metavar='DIR', help='write the TimeStep of the last timed step (rank 0) as DIR/<name>.npy')
  args = ap.parse_args()
  if args.steps < 1:
    ap.error('--steps must be at least 1')
  if args.impl == 'reference':
    run_reference(args)
  else:
    run_gpu(args)


if __name__ == '__main__':
  main()
