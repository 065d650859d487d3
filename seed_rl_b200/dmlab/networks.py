"""Policy networks on the hot path -- mirror of the reference's `dmlab/networks.py`
(`ImpalaDeep`, AgentOutput; reference dmlab/networks.py:22-171) with the same agent
protocol:

    agent.initial_state(batch_size) -> (h, c)
    agent(prev_actions, env_outputs, core_state, unroll=False, is_training=False)
        -> (AgentOutput(action, policy_logits, baseline), core_state)
    agent.get_action(...)  == agent(...)
    agent.trainable_variables  (39 tensors for ImpalaDeep, reference tests/agents_test.py:45)

All math runs in libseedrl_b200 (seedrl_net_forward / seedrl_net_backward); parameters
live in ONE flat fp32 HBM arena (Keras layouts, tf.Module variable order), which is what
the fused Adam kernel and the NCCL all-reduce operate on.  `ImpalaShallow` is the
IMPALA-paper shallow net (not in the reference, SURVEY 0), same protocol.
"""
import collections
import ctypes
import math
import threading

import numpy as np
import torch

from seed_rl_b200 import _lib

AgentOutput = collections.namedtuple('AgentOutput', 'action policy_logits baseline')

LSTM_UNITS = 256


class _CudaAgent(object):
  _NET = None

  def __init__(self, num_actions, obs_shape=(84, 84, 4), seed=0, device=None, conv_mode='simt',
               lstm_mode='tiled'):
    """conv_mode selects the arithmetic of every contraction (3x3 convs, Dense, LSTM input
    projection, policy head): 'simt' = fp32 CUDA cores (the 2e-3 parity path), 'tc' = tcgen05
    tensor cores with bf16 operands and fp32 accumulation, 'tc3' = tcgen05 with bf16x3 split
    operands (fp32-faithful)."""
    L = _lib.lib()
    self._num_actions = int(num_actions)
    self._obs_shape = tuple(int(x) for x in obs_shape)
    cfg = _lib.NetConfig(self._NET, self._num_actions, *self._obs_shape)
    h = ctypes.c_void_p()
    _lib.check(L.seedrl_net_create(ctypes.byref(cfg), ctypes.byref(h)))
    self._h = h
    modes = {'simt': 0, 'tc': 1, 'tc3': 2, 'tc3p': 3}
    if conv_mode not in modes:
      raise ValueError("conv_mode must be 'simt', 'tc' (bf16), 'tc3' (bf16x3, fp32-faithful) or "
                       "'tc3p' (bf16x3 on HBM-resident operand planes, TMA-fed)")
    if conv_mode == 'tc3p' and self._NET != _lib.NET_DEEP:
      raise ValueError("conv_mode 'tc3p' is built for the deep net")
    self.conv_mode = conv_mode
    _lib.check(L.seedrl_net_set_conv_mode(h, modes[conv_mode]))
    lstm_modes = {'stepwise': 0, 'tiled': 2}
    if lstm_mode not in lstm_modes:
      raise ValueError("lstm_mode must be 'tiled' or 'stepwise'")
    self.lstm_mode = lstm_mode
    _lib.check(L.seedrl_net_set_lstm_mode(h, lstm_modes[lstm_mode]))
    self._n_tensors = L.seedrl_net_num_param_tensors(h)
    self.arena_floats = int(L.seedrl_net_arena_floats(h))
    self.num_params = int(L.seedrl_net_num_params(h))
    self.param_info = []       # (name, shape, offset) incl. entropy_cost_param last
    for i in range(self._n_tensors + 1):
      name = ctypes.create_string_buffer(128)
      dims = (ctypes.c_int64 * 4)()
      off = ctypes.c_size_t()
      rank = L.seedrl_net_param_info(h, i, name, 128, dims, ctypes.byref(off))
      self.param_info.append((name.value.decode(), tuple(int(dims[k]) for k in range(rank)),
                              int(off.value)))
    self.device = torch.device(device if device is not None else
                               ('cuda:%d' % torch.cuda.current_device()))
    # flat arenas: params / grads (Adam slots live in the optimizer)
    self.params = torch.zeros(self.arena_floats, dtype=torch.float32, device=self.device)
    self.grads = torch.zeros_like(self.params)
    self._init_parameters(seed)
    # One activation workspace per (T1, B): the inference thread (T1=1, B=N, its own stream)
    # and the learner thread (T1=T+1, B=batch) share this agent's parameters but never a
    # workspace; backward() uses exactly the buffer its is_training forward filled.
    self._workspaces = {}
    self._lock = threading.Lock()
    self._rng_offset = 0
    self._seed = seed
    self._saved = None

  def __del__(self):
    try:
      if getattr(self, '_h', None):
        _lib.lib().seedrl_net_destroy(self._h)
        self._h = None
    except Exception:   # interpreter shutdown
      pass

  # ---- parameters ---------------------------------------------------------------
  def _view(self, arena, i):
    name, shape, off = self.param_info[i]
    n = int(np.prod(shape)) if shape else 1
    return arena[off:off + n].view(shape if shape else ())

  @property
  def trainable_variables(self):
    return [self._view(self.params, i) for i in range(self._n_tensors)]

  @property
  def variable_names(self):
    return [p[0] for p in self.param_info[:self._n_tensors]]

  def named_parameters(self):
    return collections.OrderedDict(
        (self.param_info[i][0], self._view(self.params, i)) for i in range(self._n_tensors))

  def named_gradients(self):
    return collections.OrderedDict(
        (self.param_info[i][0], self._view(self.grads, i)) for i in range(self._n_tensors + 1))

  @property
  def entropy_cost_param(self):
    return self._view(self.params, self._n_tensors)

  @property
  def entropy_cost_param_index(self):
    return self.param_info[self._n_tensors][2]

  def load_named_parameters(self, named):
    """Copies {name: array} (Keras layouts) into the arena."""
    mine = self.named_parameters()
    for k, v in named.items():
      if k == 'entropy_cost_param':
        self.entropy_cost_param.copy_(torch.as_tensor(np.asarray(v, np.float32)))
        continue
      t = torch.as_tensor(np.asarray(v, np.float32))
      if tuple(t.shape) != tuple(mine[k].shape):
        raise ValueError('shape mismatch for %s: %s vs %s' % (k, tuple(t.shape), tuple(mine[k].shape)))
      mine[k].copy_(t)

  def _init_parameters(self, seed):
    """Keras defaults (TF 2.4.1): glorot_uniform kernels, zero biases, orthogonal
    recurrent kernel, unit_forget_bias.  One-time host-side work."""
    rng = np.random.default_rng(seed)
    for i in range(self._n_tensors):
      name, shape, _ = self.param_info[i]
      if name.endswith('bias'):
        a = np.zeros(shape, np.float32)
        if name == 'core/bias':
          a[LSTM_UNITS:2 * LSTM_UNITS] = 1.0
      elif name == 'core/recurrent_kernel':
        m = rng.normal(size=(shape[1], shape[0]))
        q, r = np.linalg.qr(m)
        a = (q * np.sign(np.diag(r))).T.astype(np.float32)
      else:
        rf = int(np.prod(shape[:-2])) if len(shape) > 2 else 1
        lim = math.sqrt(6.0 / (shape[-2] * rf + shape[-1] * rf))
        a = rng.uniform(-lim, lim, shape).astype(np.float32)
      self._view(self.params, i).copy_(torch.from_numpy(a))

  # ---- protocol ---------------------------------------------------------------
  def initial_state(self, batch_size):
    z = torch.zeros([batch_size, LSTM_UNITS], dtype=torch.float32, device=self.device)
    return (z, z.clone())

  def _workspace(self, T1, B):
    key = (T1, B, threading.get_ident())
    with self._lock:
      ws = self._workspaces.get(key)
      if ws is None:
        nbytes = int(_lib.lib().seedrl_net_workspace_bytes(self._h, T1, B))
        # drop this thread's buffers of other shapes first (a learner that changes batch size
        # must not keep several multi-GB workspaces alive)
        for k in [k for k in self._workspaces if k[2] == key[2] and k != key]:
          del self._workspaces[k]
        ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        self._workspaces[key] = ws
    return ws

  def check_errors(self):
    """Raises if a kernel of the last training forward/backward hit a bounded-wait timeout
    (synchronises the current stream; call where the loss is read anyway)."""
    if self._saved is None:
      return
    T1, B, ws = self._saved[0], self._saved[1], self._saved[-1]
    _lib.check(_lib.lib().seedrl_net_check_error(self._h, T1, B, _lib.ptr(ws), ws.numel(),
                                                 _lib.stream_ptr()))

  def _next_rng_offset(self):
    with self._lock:
      o = self._rng_offset
      self._rng_offset += 1
    return o

  def get_action(self, *args, **kwargs):
    return self.__call__(*args, **kwargs)

  def __call__(self, prev_actions, env_outputs, core_state, unroll=False,
               is_training=False, gumbel_noise=None, rng_counter=None):
    """rng_counter: optional int64 CUDA scalar tensor holding the Philox offset of the sampling
    kernel; it is read and incremented ON THE DEVICE, which makes the whole call capturable in a
    CUDA graph (InferenceHost replays one graph per inference batch)."""
    reward, done, frame = env_outputs[0], env_outputs[1], env_outputs[2]
    prev_actions = _lib.require_cuda(prev_actions, torch.int64, 'prev_actions')
    reward = _lib.require_cuda(reward, torch.float32, 'reward')
    done = _lib.require_cuda(done, torch.bool, 'done')
    frame = _lib.require_cuda(frame, torch.uint8, 'observation')
    if not unroll:   # add the time dimension (networks.py:141-144)
      prev_actions, reward, done, frame = (t.unsqueeze(0) for t in (prev_actions, reward, done, frame))
    T1, B = int(prev_actions.shape[0]), int(prev_actions.shape[1])
    if tuple(frame.shape[2:]) != self._obs_shape:
      raise ValueError('observation shape %s, expected %s' % (tuple(frame.shape[2:]), self._obs_shape))
    h0 = _lib.require_cuda(core_state[0], torch.float32, 'core_state.h')
    c0 = _lib.require_cuda(core_state[1], torch.float32, 'core_state.c')
    A = self._num_actions
    logits = torch.empty([T1, B, A], dtype=torch.float32, device=self.device)
    baseline = torch.empty([T1, B], dtype=torch.float32, device=self.device)
    h = torch.empty_like(h0)
    c = torch.empty_like(c0)
    ws = self._workspace(T1, B)
    L = _lib.lib()
    st = _lib.stream_ptr()
    _lib.check(L.seedrl_net_forward(
        self._h, _lib.ptr(self.params), T1, B, _lib.ptr(prev_actions), _lib.ptr(reward),
        _lib.ptr(done), _lib.ptr(frame), _lib.ptr(h0), _lib.ptr(c0), _lib.ptr(logits),
        _lib.ptr(baseline), _lib.ptr(h), _lib.ptr(c), _lib.ptr(ws), ws.numel(), st))
    # sample a new action (networks.py:121-122)
    action = torch.empty([T1 * B], dtype=torch.int64, device=self.device)
    noise = None
    if gumbel_noise is not None:
      noise = _lib.require_cuda(gumbel_noise, torch.float32, 'gumbel_noise')
    if rng_counter is not None:
      _lib.check(L.seedrl_categorical_sample_counter(
          T1 * B, A, _lib.ptr(logits), _lib.ptr(noise), int(self._seed), _lib.ptr(rng_counter), _lib.ptr(action), st))
    else:
      _lib.check(L.seedrl_categorical_sample(
          T1 * B, A, _lib.ptr(logits), _lib.ptr(noise), int(self._seed), int(self._next_rng_offset()),
          _lib.ptr(action), st))
    action = action.view(T1, B)
    if is_training:
      self._saved = (T1, B, prev_actions, reward, done, frame, ws)
    out = AgentOutput(action, logits, baseline)
    if not unroll:
      out = AgentOutput(*(t.squeeze(0) for t in out))
    return out, (h, c)

  def backward(self, dlogits, dbaseline, head_ready_event=None):
    """d loss / d parameters for the last is_training unroll -> self.grads (overwritten).
    head_ready_event: a torch.cuda.Event recorded once grads[:self.grad_split] (heads, Dense,
    LSTM) are final -- before the convolution torso's backward -- for an overlapped all-reduce."""
    if self._saved is None:
      raise RuntimeError('backward() needs a preceding __call__(..., unroll=True, is_training=True)')
    T1, B, prev_actions, reward, done, frame, ws = self._saved
    L = _lib.lib()
    if head_ready_event is None:
      _lib.check(L.seedrl_net_backward(
          self._h, _lib.ptr(self.params), T1, B, _lib.ptr(prev_actions), _lib.ptr(reward),
          _lib.ptr(done), _lib.ptr(frame), _lib.ptr(dlogits), _lib.ptr(dbaseline),
          _lib.ptr(self.grads), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()))
    else:
      head_ready_event.record()        # creates the underlying cudaEvent_t; re-recorded by the library
      _lib.check(L.seedrl_net_backward_overlap(
          self._h, _lib.ptr(self.params), T1, B, _lib.ptr(prev_actions), _lib.ptr(reward),
          _lib.ptr(done), _lib.ptr(frame), _lib.ptr(dlogits), _lib.ptr(dbaseline),
          _lib.ptr(self.grads), _lib.ptr(ws), ws.numel(), ctypes.c_void_p(head_ready_event.cuda_event),
          _lib.stream_ptr()))
    return self.grads

  @property
  def grad_split(self):
    return int(_lib.lib().seedrl_net_grad_split(self._h))

  # learner.py:225-234 adds these to the agent when it has no entropy_cost()
  def init_entropy_cost(self, entropy_cost, adjustment_speed):
    self._entropy_mul = float(adjustment_speed)
    self.entropy_cost_param.fill_(math.log(entropy_cost) / adjustment_speed)

  def entropy_cost(self):
    return torch.exp(self._entropy_mul * self.entropy_cost_param)

  def state_dict(self):
    return {'params': self.params.detach().cpu(), 'param_info': self.param_info}

  def load_state_dict(self, d):
    self.params.copy_(d['params'].to(self.device))


class ImpalaDeep(_CudaAgent):
  """reference dmlab/networks.py:63-171."""
  _NET = _lib.NET_DEEP


class ImpalaShallow(_CudaAgent):
  """IMPALA-paper shallow net: conv 8x8/4 ->16, conv 4x4/2 ->32, FC 256, LSTM 256."""
  _NET = _lib.NET_SHALLOW
