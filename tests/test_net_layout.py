"""CPU: the parameter arenas and activation workspaces of the network schedules (csrc/net.cu,
csrc/r2d2_net.cu) are pinned -- every tensor's name, dims and offset, the arena size, the gradient
bucket split and the workspace size for a few unroll shapes per conv mode.  Checkpoints, the
all-reduce buckets and callers' workspace allocations depend on them; tests/golden/net_layout.json
holds the values."""
import ctypes
import json
import os

import pytest

from seed_rl_b200 import _lib

GOLDEN = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'net_layout.json')))


def _name(e):
  return '%s-%dx%dx%d' % ((e.get('net', 'r2d2'),) + tuple(e['obs']))


def _param_table(count, info):
  out = []
  for i in range(count):
    name = ctypes.create_string_buffer(128)
    dims = (ctypes.c_int64 * 4)()
    off = ctypes.c_size_t()
    rank = info(i, name, dims, off)
    out.append([name.value.decode(), [int(dims[k]) for k in range(rank)], int(off.value)])
  return out


@pytest.mark.parametrize('g', GOLDEN['impala'], ids=_name)
def test_impala_net_layout(g):
  L = _lib.lib()
  h = ctypes.c_void_p()
  cfg = _lib.NetConfig(_lib.NET_DEEP if g['net'] == 'deep' else _lib.NET_SHALLOW, g['num_actions'], *g['obs'])
  _lib.check(L.seedrl_net_create(ctypes.byref(cfg), ctypes.byref(h)))
  try:
    params = _param_table(L.seedrl_net_num_param_tensors(h) + 1,       # + entropy_cost_param
                          lambda i, name, dims, off: L.seedrl_net_param_info(h, i, name, 128, dims, ctypes.byref(off)))
    assert params == g['params']
    assert L.seedrl_net_arena_floats(h) == g['arena_floats']
    assert L.seedrl_net_grad_split(h) == g['grad_split']
    for mode, sizes in g['workspace_bytes'].items():
      _lib.check(L.seedrl_net_set_conv_mode(h, int(mode)))
      for T1, B, want in sizes:
        assert L.seedrl_net_workspace_bytes(h, T1, B) == want, (mode, T1, B)
  finally:
    L.seedrl_net_destroy(h)


@pytest.mark.parametrize('g', GOLDEN['r2d2'], ids=_name)
def test_r2d2_net_layout(g):
  L = _lib.lib()
  h = ctypes.c_void_p()
  _lib.check(L.seedrl_r2d2_net_create(g['num_actions'], *g['obs'], ctypes.byref(h)))

  def info(i, name, dims, off):
    rank = ctypes.c_int()
    _lib.check(L.seedrl_r2d2_net_param_info(h, i, name, 128, dims, ctypes.byref(rank), ctypes.byref(off)))
    return rank.value
  try:
    assert _param_table(L.seedrl_r2d2_net_num_param_tensors(h), info) == g['params']
    assert L.seedrl_r2d2_net_arena_floats(h) == g['arena_floats']
    for T, B, want in g['workspace_bytes']:
      assert L.seedrl_r2d2_net_workspace_bytes(h, T, B) == want, (T, B)
  finally:
    L.seedrl_r2d2_net_destroy(h)


def test_r2d2_workspace_holds_the_stepwise_lstm_buffers():
  """The R2D2 workspace has room for the per-step LSTM schedule: the dh(t-1) and the two
  alternating dc buffers of the stepwise BPTT, three B x 512 fp32 arrays, on top of the
  8 121 853 696 bytes the tiled recurrence alone needs at T = 141, B = 64 (84x84x4 frames)."""
  L = _lib.lib()
  h = ctypes.c_void_p()
  _lib.check(L.seedrl_r2d2_net_create(18, 84, 84, 4, ctypes.byref(h)))
  try:
    assert L.seedrl_r2d2_net_workspace_bytes(h, 141, 64) == 8121853696 + 3 * 64 * 512 * 4 == 8122246912
  finally:
    L.seedrl_r2d2_net_destroy(h)


def test_lstm_mode_is_stepwise_or_tiled():
  """lstm_mode 0 = a GEMM + a pointwise kernel per step, 2 = the tiled persistent kernels; 1 named
  an earlier persistent form and is refused."""
  L = _lib.lib()
  h = ctypes.c_void_p()
  cfg = _lib.NetConfig(_lib.NET_SHALLOW, 6, 84, 84, 4)
  _lib.check(L.seedrl_net_create(ctypes.byref(cfg), ctypes.byref(h)))
  r = ctypes.c_void_p()
  _lib.check(L.seedrl_r2d2_net_create(6, 36, 36, 4, ctypes.byref(r)))
  try:
    for set_mode, net in ((L.seedrl_net_set_lstm_mode, h), (L.seedrl_r2d2_net_set_lstm_mode, r)):
      for mode in (0, 2):
        _lib.check(set_mode(net, mode))
      for mode in (1, 3, -1):
        assert set_mode(net, mode) == 3        # SEEDRL_ERR_INVALID_ARGUMENT
  finally:
    L.seedrl_net_destroy(h)
    L.seedrl_r2d2_net_destroy(r)
