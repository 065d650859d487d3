"""GPU: the central-inference path (a6/a7/a8/a9): InferenceHost._inference ==
reference agents/vtrace/learner.py:351-405 -- run-id resets, T=1 forward + sampling,
UnrollStore append, first-state bookkeeping, capacity-1 queue, time-major batch assembly;
then served end to end through the RPC server + C++ batcher."""
import threading

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

A, OBS = 18, (84, 84, 4)


def _host(num_envs, T, N):
  from seed_rl_b200.agents.vtrace import learner_loop
  from seed_rl_b200.dmlab import networks
  agent = networks.ImpalaDeep(A, OBS, seed=3)
  return learner_loop.InferenceHost(agent, num_envs, T, N, OBS), agent


def _env_batch(rng, ids, step):
  from seed_rl_b200.common import utils
  n = len(ids)
  return utils.EnvOutput(
      rng.normal(size=n).astype(np.float32), rng.random(n) < 0.15,
      rng.integers(0, 256, (n,) + OBS, dtype=np.uint8), np.zeros(n, bool),
      np.full(n, step, np.int32))


def test_inference_unrolls_are_consistent_with_training_unroll():
  from seed_rl_b200.agents.vtrace import learner_loop
  num_envs, T, N = 6, 3, 3
  host, agent = _host(num_envs, T, N)
  got, stop = [], threading.Event()

  def consumer():
    from seed_rl_b200.common import utils
    while True:
      try:
        got.append(host.unroll_queue.dequeue())
      except utils.QueueClosedError:
        return
  th = threading.Thread(target=consumer); th.start()
  rng = np.random.default_rng(0)
  run_ids = rng.integers(1, 2**40, num_envs)
  actions_seen = {e: [] for e in range(num_envs)}
  for step in range(9):
    for ids in (np.array([0, 1, 2], np.int32), np.array([5, 3, 4], np.int32)):
      env = _env_batch(rng, ids, step)
      act = host.inference(ids, run_ids[ids], env, np.zeros(len(ids), np.float32))
      assert act.shape == (3,) and act.dtype == np.int64 and (0 <= act).all() and (act < A).all()
      for e, a in zip(ids, act):
        actions_seen[int(e)].append(int(a))
  torch.cuda.synchronize()
  host.unroll_queue.close(); th.join(10)
  # 9 steps, unroll length 3 (+1 overlap row): unrolls complete at steps 4 and 7 -> 2 per env
  assert len(got) == 2 * num_envs
  for u in got:
    T1 = T + 1
    assert tuple(u.prev_actions.shape) == (T1,) and tuple(u.env_outputs.observation.shape) == (T1,) + OBS
    # the action produced at step t is the prev_action of step t+1 (learner.py:402-403)
    assert torch.equal(u.agent_outputs.action[:-1], u.prev_actions[1:])
    # replay through the training-mode unroll from the stored first state
    batch = learner_loop.dequeue_batch(_OneShot(u), 1)
    out, _ = agent(batch.prev_actions, batch.env_outputs, batch.agent_state, unroll=True)
    np.testing.assert_allclose(out.policy_logits[:, 0].cpu().numpy(),
                               u.agent_outputs.policy_logits.cpu().numpy(), rtol=2e-4, atol=2e-5)
    np.testing.assert_allclose(out.baseline[:, 0].cpu().numpy(),
                               u.agent_outputs.baseline.cpu().numpy(), rtol=2e-4, atol=2e-5)
  # a new run id resets the env's store/state (learner.py:353-366): next unroll needs T+1 steps again
  ids = np.array([0, 1, 2], np.int32)
  new_run = run_ids.copy(); new_run[0] += 1
  host.unroll_queue = type(host.unroll_queue)(-1, host.unroll_specs)
  for step in range(T):
    host.inference(ids, new_run[ids], _env_batch(rng, ids, step), np.zeros(3, np.float32))
  # envs 1,2 were at index 1 (carry row) and complete after T more steps; env 0 was reset
  assert host.unroll_queue.size() == 2


class _OneShot(object):
  def __init__(self, u):
    self.u = u

  def dequeue(self):
    return self.u


def test_time_major_batch_assembly_matches_make_time_major():
  """dequeue_batch == stack + make_time_major of the reference (learner.py:418-432)."""
  from seed_rl_b200.agents.vtrace import learner_loop
  from seed_rl_b200.common import utils
  rng = np.random.default_rng(1)
  T1, B = 4, 3
  mk = lambda *s, dt=np.float32: torch.as_tensor(rng.normal(size=s).astype(dt)).cuda()
  unrolls = []
  from seed_rl_b200.dmlab import networks
  for _ in range(B):
    env = utils.EnvOutput(mk(T1), mk(T1) > 0, (mk(T1, 5, 5, 4) * 50).to(torch.uint8), mk(T1) > 9, mk(T1).int())
    ao = networks.AgentOutput(mk(T1).long(), mk(T1, A), mk(T1))
    unrolls.append(learner_loop.Unroll((mk(256), mk(256)), mk(T1).long(), env, ao))

  class Q(object):
    def __init__(self): self.i = 0
    def dequeue(self):
      self.i += 1
      return unrolls[self.i - 1]
  b = learner_loop.dequeue_batch(Q(), B)
  ref = utils.make_time_major(utils.map_structure(lambda *xs: torch.stack(xs), *[u[1:] for u in unrolls]))
  for x, y in zip(utils.flatten(b[1:]), utils.flatten(ref)):
    assert torch.equal(x, y)
  assert tuple(b.agent_state[0].shape) == (B, 256)
  assert tuple(b.env_outputs.observation.shape) == (T1, B, 5, 5, 4)


def test_served_through_rpc_and_batcher(tmp_path):
  """Actors -> gRPC -> pinned-slab batcher -> GPU inference -> actions back."""
  from seed_rl_b200.grpc import ops
  # two actors with [2]-slices into batches of 4: they always pair with each other, so no
  # partially filled batch can be left waiting (which blocks forever, as in the reference).
  num_envs, T, N = 4, 2, 4
  host, agent = _host(num_envs, T, N)
  host.unroll_queue = type(host.unroll_queue)(-1, host.unroll_specs)   # nobody trains here
  address = 'unix:%s' % (tmp_path / 'sock')
  server = ops.Server([address])
  server.bind(host.inference)
  server.start()
  rng = np.random.default_rng(2)
  results = {}

  def actor(k):           # env_batch_size 2: each actor contributes [2] slices
    c = ops.Client(address)
    ids = np.array([2 * k, 2 * k + 1], np.int32)
    run = rng.integers(1, 2**40, 2)
    out = []
    for step in range(T + 1):
      env = _env_batch(np.random.default_rng(10 * k + step), ids, step)
      out.append(c.inference(ids, run, env, np.zeros(2, np.float32)))
    results[k] = out
  ts = [threading.Thread(target=actor, args=(k,)) for k in range(2)]
  [t.start() for t in ts]; [t.join(60) for t in ts]
  server.shutdown()
  assert sorted(results) == [0, 1]
  for out in results.values():
    assert all(o.shape == (2,) and o.dtype == np.int64 for o in out)
  assert host.unroll_queue.size() == num_envs      # every env completed one unroll


def test_device_feeder_double_buffering():
  """learner.DeviceFeeder: batches come out in order with the uploaded contents; a third put
  without a get is refused; a slot is only overwritten after its consumer was marked done."""
  from seed_rl_b200.agents.vtrace import learner
  mk = lambda v: {'a': torch.full((1 << 20,), float(v)).pin_memory(), 'b': torch.full((3, 5), v, dtype=torch.int64).pin_memory()}
  f = learner.DeviceFeeder(mk(0))
  f.put(mk(1)); f.put(mk(2))
  with pytest.raises(RuntimeError):
    f.put(mk(3))
  seen = []
  for nxt in (3, 4, 5, None, None):
    slot, d = f.get()
    acc = d['a'].sum() / d['a'].numel() + d['b'].float().mean()     # consume on the compute stream
    f.done_with(slot)
    if nxt is not None:
      f.put(mk(nxt))
    seen.append(float(acc))
  assert seen == [2.0, 4.0, 6.0, 8.0, 10.0]
  with pytest.raises(RuntimeError):
    f.get()


def test_zero_copy_batch_assembly_matches_queue_path():
  """SURVEY 8(f) rank 2: the assembler path (completed unrolls gathered straight into columns of
  the time-major training batch; no per-unroll tensors, no stack, no host read-back of the
  completion count) yields bit-identical training batches to the reference-shaped path (capacity-1
  queue of single unrolls + dequeue_batch), including batches that straddle inference calls."""
  from seed_rl_b200.agents.vtrace import learner_loop
  from seed_rl_b200.common import utils
  from seed_rl_b200.dmlab import networks
  num_envs, T, N, B = 6, 3, 3, 4
  agent = networks.ImpalaDeep(A, OBS, seed=3)
  host_q = learner_loop.InferenceHost(agent, num_envs, T, N, OBS)
  host_q.unroll_queue = type(host_q.unroll_queue)(-1, host_q.unroll_specs)
  host_a = learner_loop.InferenceHost(agent, num_envs, T, N, OBS, training_batch_size=B)
  # same sampling noise on both hosts: the agent's RNG offset advances per call, so replay it
  rng = np.random.default_rng(0)
  run_ids = rng.integers(1, 2**40, num_envs)
  calls = []
  for step in range(9):
    for ids in (np.array([0, 1, 2], np.int32), np.array([5, 3, 4], np.int32)):
      calls.append((ids, _env_batch(rng, ids, step)))
  batches_a = []

  def learner_thread():
    try:
      while True:
        slot, u = learner_loop.assembled_batch(host_a.assembler)
        batches_a.append(utils.map_structure(lambda t: t.clone(), tuple(u)))
        host_a.assembler.release(slot)
    except utils.QueueClosedError:
      return
  th = threading.Thread(target=learner_thread); th.start()
  for host in (host_q, host_a):
    agent._rng_offset = 0
    for ids, env in calls:
      host.inference(ids, run_ids[ids], env, np.zeros(len(ids), np.float32))
  torch.cuda.synchronize()
  import time
  for _ in range(100):
    if len(batches_a) == 3:
      break
    time.sleep(0.05)
  host_a.assembler.close(); th.join(10)
  assert host_q.unroll_queue.size() == 12 and len(batches_a) == 3      # 12 unrolls = 3 batches of 4
  assert host_a.store._host_index is not None                          # completion tracked on the host
  for k in range(3):
    want = learner_loop.dequeue_batch(host_q.unroll_queue, B)
    for x, y in zip(utils.flatten(batches_a[k]), utils.flatten(tuple(want))):
      assert torch.equal(x, y)
