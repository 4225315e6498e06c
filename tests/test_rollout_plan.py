"""Host side of the persistent rollout kernel (csrc/rollout_fused.cu): the shared-memory plan that decides whether a policy
is taken by the kernel or the actors keep the per-step launch sequence.  No GPU needed: planning is host code behind the
C-ABI (`sb200_ppo_rollout_supported`)."""
import ctypes as C

import pytest

from surreal_b200 import _lib, ops


def _supported(dims):
    A = dims[-1]
    net = ops.FlatNet(dims, [ops.ACT_RELU] * (len(dims) - 2) + [ops.ACT_TANH], 'cpu', extra=A)
    return bool(_lib.lib().sb200_ppo_rollout_supported(C.byref(net.desc()), dims[0], A))


@pytest.mark.parametrize('dims', [
    [64, 256, 256, 8],          # the benchmark's policy
    [12, 48, 32, 3],            # the per-step comparison tests
    [12, 96, 64, 32],           # heads whose slice sums need more of the Part buffer than the hidden layers' tiles
    [64, 16, 16, 8],
])
def test_policies_the_kernel_takes(dims):
    assert _supported(dims)


@pytest.mark.parametrize('dims', [
    [66, 256, 256, 8],          # observations move as float4: D % 4 == 0
    [132, 256, 256, 8],         # one float4 of the input tile per lane: D <= 128
    [64, 40, 256, 8],           # four CTAs x column quads: hidden widths % 16 == 0
    [64, 256, 256, 33],         # one lane per action: A <= 32
    [64, 128, 128, 128, 8],     # exactly two hidden layers
    [64, 512, 256, 8],          # resident weights and tiles over 224 KB of shared memory
])
def test_policies_the_kernel_rejects(dims):
    assert not _supported(dims)
