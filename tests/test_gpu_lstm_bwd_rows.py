"""The backward recurrence (csrc/lstm.cu) has a row-split form (lstm_bwd_rows_kernel: the batch rows split between two
halves of the grid, clusters of 4 CTAs owning 64 units each) next to the unsplit cluster form (lstm_bwd_cluster_kernel,
clusters of 4 CTAs owning 32 units for all rows).  Each warp contracts the same k-slice in the same MMA order and the
partial sums meet in the same order, so the dgates buffer must be bit-identical; the gradients downstream of it go
through GEMMs that may split K and are compared within the tolerance of test_lstm_backward_variants_agree."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SWITCHES = ("VQA_B200_LSTM_BWD_ROWS", "VQA_B200_LSTM_BWD_CLUSTER")
SPLIT = {"VQA_B200_LSTM_BWD_ROWS": "2"}
UNSPLIT = {"VQA_B200_LSTM_BWD_ROWS": "1", "VQA_B200_LSTM_BWD_CLUSTER": "4"}


class _env:
    """Sets the launch-form switches (read by the library at every launch) for the duration of a block."""

    def __init__(self, env):
        self.env = env

    def __enter__(self):
        for k in SWITCHES:
            os.environ.pop(k, None)
        os.environ.update(self.env)

    def __exit__(self, *exc):
        for k in SWITCHES:
            os.environ.pop(k, None)


def _inputs(S, Bt, H, seed):
    g = torch.Generator().manual_seed(seed)
    pre = torch.randn(S, Bt, 4, H, generator=g)
    gates = torch.cat([torch.sigmoid(pre[:, :, :2]), torch.tanh(pre[:, :, 2:3]), torch.sigmoid(pre[:, :, 3:])], 2)
    c_all = torch.randn(S, Bt, H, generator=g)
    dout = torch.randn(Bt, S, H, generator=g)                  # the caller's [Bt, S, H] order, read through strides
    whh = ((torch.rand(4 * H, H, generator=g) * 2 - 1) * (6.0 / (5 * H)) ** 0.5).to(torch.bfloat16)
    return [t.to(DEV) for t in (gates.reshape(S, Bt, 4 * H).contiguous(), c_all, dout, whh)]


def _bwd(inputs, S, Bt, H, drop_p, env):
    from vqa_attention_networks_b200 import ops
    gates, c_all, dout, whh = inputs
    dg = ops._sentinel_bf16((S * Bt, 4 * H), DEV)
    with _env(env):
        ops._call("vqa_b200_lstm_bwd", "lstm_bwd", ops._p(gates), ops._p(c_all), ops._p(dout), dout.stride(1),
                  dout.stride(0), ops._p(whh), 1, ops._p(dg), S, Bt, H, float(drop_p), 4321, None, ops._st())
        torch.cuda.synchronize()
    return dg.view(torch.int16)


@pytest.mark.parametrize("H", [128, 256, 512, 1024])
@pytest.mark.parametrize("Bt", [1, 2, 7, 13, 26, 32])
@pytest.mark.parametrize("S", [1, 2, 256])
@pytest.mark.parametrize("drop_p", [0.0, 0.3])
def test_backward_row_split_dgates_bit_equal(H, Bt, S, drop_p):
    inputs = _inputs(S, Bt, H, 10 * H + Bt + S)
    ref = _bwd(inputs, S, Bt, H, drop_p, UNSPLIT)
    assert not (ref == -1).any()                      # every step published
    got = _bwd(inputs, S, Bt, H, drop_p, SPLIT)
    assert torch.equal(got, ref)


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


@pytest.mark.parametrize("Bt,S,E,H", [(5, 6, 24, 128), (20, 9, 40, 256), (32, 17, 64, 512), (26, 48, 300, 1024),
                                      (2, 200, 300, 1024)])
def test_backward_row_split_gradients_agree(Bt, S, E, H):
    from vqa_attention_networks_b200 import ops
    g = torch.Generator().manual_seed(77)
    x = torch.tanh(torch.randn(Bt, S, E, generator=g))
    W_ih = (torch.rand(4 * H, E, generator=g) * 2 - 1) * (6.0 / (4 * H + E)) ** 0.5
    W_hh = (torch.rand(4 * H, H, generator=g) * 2 - 1) * (6.0 / (5 * H)) ** 0.5
    b_ih, b_hh = [(torch.rand(4 * H, generator=g) * 2 - 1) * H ** -0.5 for _ in range(2)]
    cot = torch.randn(Bt, S, H, generator=g).to(DEV)
    grads = []
    for env in (UNSPLIT, SPLIT):
        xg = x.to(DEV).requires_grad_(True)
        pg = [p.to(DEV).requires_grad_(True) for p in (W_ih, W_hh, b_ih, b_hh)]
        with _env(env):
            out = ops.LstmFn.apply(xg, *pg, ops.WeightCache())
            out.backward(cot)
            torch.cuda.synchronize()
        grads.append([xg.grad] + [p.grad for p in pg])
    for a, b in zip(*grads):
        assert _rel(a, b) <= 1e-3


def test_row_split_setting_is_checked():
    inputs = _inputs(2, 3, 128, 0)
    with pytest.raises(RuntimeError, match="VQA_B200_LSTM_BWD_ROWS"):
        _bwd(inputs, 2, 3, 128, 0.0, {"VQA_B200_LSTM_BWD_ROWS": "3"})
