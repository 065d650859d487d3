"""The tiled persistent LSTM recurrence (csrc/lstm_tiled.cu: one launch for all T steps, each way;
CTA = (batch tile, 16 hidden units)) against the per-step schedule (a GEMM + a pointwise kernel per
step), on the same agent and inputs, for both nets that share the LSTM core (csrc/net_common.cu):
LSTMCell(256) of the IMPALA nets (dmlab/networks.py:157-169) and LSTMCell(512) of the R2D2 net
(atari/networks.py:240-252).  Both schedules are fp32 throughout; they differ in summation order
only."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _impala_shallow(T, B):
  """Same logits, state and loss to 1e-5, gradients to 1e-4 of each tensor's max."""
  from oracle import learner_oracle
  from seed_rl_b200.agents.vtrace import learner
  from seed_rl_b200.common import optimizers
  from seed_rl_b200.dmlab import networks
  from test_gpu_parity import _batch_to_cuda
  A, OBS = 18, (84, 84, 4)
  b = learner_oracle.synthetic_batch(T, B, A, seed=5)
  b['done'][min(1, T), 0] = True
  rng = np.random.default_rng(1)
  b['h0'] = rng.normal(size=b['h0'].shape).astype(np.float32)
  b['c0'] = rng.normal(size=b['c0'].shape).astype(np.float32)
  u = _batch_to_cuda(b)
  res = {}
  for mode in ('stepwise', 'tiled'):
    agent = networks.ImpalaShallow(A, OBS, seed=2, lstm_mode=mode)    # cheap torso, same LSTM
    step = learner.LearnerStep(agent, optimizers.Adam(1e-3))
    out, (h, c) = agent(u.prev_actions, u.env_outputs, u.agent_state, unroll=True)
    loss, _ = step.compute_gradients(u)
    res[mode] = (out.policy_logits.clone(), h.clone(), c.clone(), float(loss),
                 {k: v.clone() for k, v in agent.named_gradients().items()})
  a, p = res['stepwise'], res['tiled']
  for i in range(3):
    np.testing.assert_allclose(p[i].cpu().numpy(), a[i].cpu().numpy(), rtol=1e-5, atol=1e-5)
  assert abs(a[3] - p[3]) < 1e-5 * max(1.0, abs(a[3]))
  for k in a[4]:
    x, y = p[4][k].cpu().numpy(), a[4][k].cpu().numpy()
    assert np.abs(x - y).max() <= 1e-4 * (np.abs(y).max() + 1e-12), k


def _r2d2(T, B):
  """Same q-values and state to 2e-5 of each tensor's max, gradients to 1e-4 relative L2.  The tiled
  kernel computes in fp32 in every GEMM mode; 'simt' keeps the stepwise recurrent product in fp32
  too (in 'tc3' it would run on the tensor cores with bf16x3 operands for B >= 64)."""
  from oracle import r2d2_learner_oracle as RL
  from seed_rl_b200 import _lib
  from seed_rl_b200.atari import networks
  from seed_rl_b200.common import utils
  A, obs, S = 6, (36, 36, 1), 4
  b = RL.synthetic_replay_batch(T, B, A, obs, seed=B, done_p=0.2)
  c = lambda a: torch.as_tensor(np.asarray(a)).cuda()
  env = utils.EnvOutput(c(b['reward']), c(b['done']), c(b['observation']),
                        torch.zeros(T, B, dtype=torch.bool).cuda(), torch.zeros(T, B, dtype=torch.int32).cuda())
  state = networks.AgentState((c(b['h0']), c(b['c0'])), c(b['frame_state']))
  agent = networks.DuelingLSTMDQNNet(A, obs, S, seed=11, gemm_mode='simt')
  dq = torch.randn(T, B, A, device='cuda', generator=torch.Generator(device='cuda').manual_seed(2))
  res = {}
  for mode in (0, 2):                        # 0 = stepwise, 2 = tiled (the default)
    _lib.check(_lib.lib().seedrl_r2d2_net_set_lstm_mode(agent._h, mode))
    out, st = agent((c(b['prev_actions']), env), state, unroll=True, is_training=True)
    agent.backward(dq)
    agent.check_errors()
    res[mode] = (out.q_values.clone(), st.core_state[0].clone(), st.core_state[1].clone(), agent.grads.clone())
  for x, y in zip(res[2][:3], res[0][:3]):
    scale = float(y.abs().max()) + 1e-30
    assert float((x - y).abs().max()) <= 2e-5 * scale, float((x - y).abs().max()) / scale
  # gradients: L2 (a head unit within rounding of its ReLU kink may flip between the two summation orders)
  gx, gy = res[2][3].double(), res[0][3].double()
  assert float((gx - gy).norm() / gy.norm()) <= 1e-4


@pytest.mark.parametrize('net,T,B',
                         [('impala_shallow', T, B) for T, B in [(6, 5), (3, 70), (1, 3), (20, 64), (5, 256), (4, 300)]] +
                         [('r2d2', T, B) for T, B in [(5, 40), (3, 64), (4, 9), (2, 100)]])
def test_tiled_lstm_matches_stepwise_schedule(net, T, B):
  (_impala_shallow if net == 'impala_shallow' else _r2d2)(T, B)
