"""The strided 'valid' convolutions of the IMPALA shallow net (dmlab/networks.py:60-75 of the paper's
small net; reference agents use it via atari/dmlab configs) and of the R2D2 body
(atari/networks.py:228-238) run as GEMMs whose im2col operand is gathered from the NHWC input while
the operand blocks are staged (csrc/gemm_tc_kernels.cu, ConvGather).  The gathered and the
materialised operand feed the tensor cores the same bf16 units in the same order, so the two
schedules must agree BIT FOR BIT -- forward outputs and every gradient tensor."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _ab(run):
  from seed_rl_b200 import _lib
  L = _lib.lib()
  res = {}
  try:
    for g in (1, 0):
      _lib.check(L.seedrl_debug_set_gemm_gather(g))
      n0 = _lib.launch_count()
      res[g] = run()
      torch.cuda.synchronize()
      res[g] = tuple(t.clone() for t in res[g]) + (_lib.launch_count() - n0,)
  finally:
    _lib.check(L.seedrl_debug_set_gemm_gather(1))
  return res


@pytest.mark.parametrize('T,B,obs,S', [(6, 8, (84, 84, 1), 4), (3, 5, (44, 40, 4), 1), (2, 70, (84, 84, 1), 4)])
def test_r2d2_body_gathered_equals_materialised(T, B, obs, S):
  from oracle import r2d2_learner_oracle as RL
  from seed_rl_b200.atari import networks
  from seed_rl_b200.common import utils
  A = 18
  b = RL.synthetic_replay_batch(T, B, A, obs, seed=T + B, done_p=0.1)
  c = lambda a: torch.as_tensor(np.asarray(a)).cuda()
  env = utils.EnvOutput(c(b['reward']), c(b['done']), c(b['observation']),
                        torch.zeros(T, B, dtype=torch.bool).cuda(), torch.zeros(T, B, dtype=torch.int32).cuda())
  state = networks.AgentState((c(b['h0']), c(b['c0'])), c(b['frame_state']) if S > 1 else ())
  agent = networks.DuelingLSTMDQNNet(A, obs, S, seed=3, gemm_mode='tc3')
  dq = torch.randn(T, B, A, device='cuda', generator=torch.Generator(device='cuda').manual_seed(1))

  def run():
    out, st = agent((c(b['prev_actions']), env), state, unroll=True, is_training=True)
    agent.backward(dq)
    agent.check_errors()
    return out.q_values, st.core_state[0], agent.grads
  r = _ab(run)
  assert r[1][-1] < r[0][-1]                 # the gathered schedule launches no im2col kernels
  for x, y in zip(r[1][:-1], r[0][:-1]):
    assert torch.equal(x, y)
  assert float(r[1][2].abs().max()) > 0


@pytest.mark.parametrize('mode', ['tc', 'tc3'])
@pytest.mark.parametrize('T,B', [(4, 3), (20, 16)])
def test_shallow_net_gathered_equals_materialised(mode, T, B):
  from oracle import learner_oracle
  from seed_rl_b200.agents.vtrace import learner
  from seed_rl_b200.common import optimizers, utils
  from seed_rl_b200.dmlab import networks
  A = 18
  agent = networks.ImpalaShallow(A, (84, 84, 4), seed=5, conv_mode=mode)
  b = learner_oracle.synthetic_batch(T, B, A, seed=7)
  c = lambda a: torch.as_tensor(np.asarray(a)).cuda()
  T1 = T + 1
  env = utils.EnvOutput(c(b['reward']), c(b['done']), c(b['observation']),
                        torch.zeros(T1, B, dtype=torch.bool).cuda(), torch.zeros(T1, B, dtype=torch.int32).cuda())
  ao = networks.AgentOutput(c(b['action']), c(b['behaviour_logits']), c(b['behaviour_baseline']))
  u = learner.Unroll((c(b['h0']), c(b['c0'])), c(b['prev_actions']), env, ao)
  step = learner.LearnerStep(agent, optimizers.Adam(1e-4), settings=learner.default_loss_settings())

  def run():
    loss, _ = step.compute_gradients(u)
    agent.check_errors()
    return loss.reshape(1), agent.grads
  r = _ab(run)
  assert r[1][-1] < r[0][-1]
  for x, y in zip(r[1][:-1], r[0][:-1]):
    assert torch.equal(x, y)
  assert float(r[1][1].abs().max()) > 0

