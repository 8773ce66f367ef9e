"""Two GPUs in one process: the tensor-core linear and the fused decoder chain, which opt into more than 48 KB of
dynamic shared memory, run on cuda:1 after they ran on cuda:0 and give the same results there.  A kernel's
shared-memory limit is held per device, so the opt-in has to happen on each device a process launches on."""
import numpy as np
import pytest
import torch

from tests import chain_cases as CC

pytestmark = pytest.mark.gpu


def _run(ops, dev):
    g = torch.Generator().manual_seed(5)
    R = 300
    A = torch.randn((R, CC.D), generator=g)
    W = torch.randn((CC.F, CC.D), generator=g) / 11
    b = torch.randn((CC.F,), generator=g)
    P = CC.gauss_params(7)
    attn = np.random.default_rng(1).standard_normal((R, CC.D)).astype(np.float32)
    x = np.random.default_rng(2).standard_normal((R, CC.D)).astype(np.float32)
    with torch.cuda.device(dev):
        d = lambda a: torch.as_tensor(a).to(dev)
        Pd = {k: d(v) for k, v in P.items()}
        y = ops.linear_tc(d(A), ops.linear_prepare(d(W)), CC.F, d(b))
        prep = ops.decoder_chain_prepare(Pd["Wo"], Pd["W1"], Pd["W2"], Pd["Win"])
        x_out, qkv = ops.decoder_chain_tc(d(attn), d(x), prep, Pd["bo"], Pd["g1"], Pd["b1"], Pd["c2"], Pd["g2"], Pd["b2"],
                                          Pd["bf1"], Pd["bf2"], Pd["g3"], Pd["b3"], Pd["bin"])
        torch.cuda.synchronize()
        assert int(ops._error_flag(torch.device(dev)).item()) == 0
    return y.cpu(), x_out.cpu(), qkv.cpu()


def test_linear_and_chain_on_two_devices():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 visible CUDA devices")
    from influentialrs_b200 import ops
    first = _run(ops, "cuda:0")
    second = _run(ops, "cuda:1")
    for a, b in zip(first, second):
        assert torch.equal(a, b)
