"""The backward recurrence (csrc/lstm.cu) runs in its row-split form by default (lstm_bwd_rows_kernel: the batch rows
split between two halves of the grid, clusters of 4 CTAs owning 64 units each; at Bt = 1 the first half only).  The rows
of a batch are independent recurrences and the kernel computes a row's element the same way whichever half and m-tile
row it sits in, so the dgates of a batched run must be bit-identical to running each row alone as a Bt = 1 problem.
That catches wrong half offsets, canaries on the wrong row, leakage across the halves and any difference between the
Bt = 1 grid and the split grid.  The gradients downstream of dgates, and the single-CTA form, are compared in
tests/test_gpu_lstm.py::test_lstm_backward_variants_agree."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SEED = 4321


def _inputs(S, Bt, H, seed):
    g = torch.Generator().manual_seed(seed)
    pre = torch.randn(S, Bt, 4, H, generator=g)
    gates = torch.cat([torch.sigmoid(pre[:, :, :2]), torch.tanh(pre[:, :, 2:3]), torch.sigmoid(pre[:, :, 3:])], 2)
    c_all = torch.randn(S, Bt, H, generator=g)
    dout = torch.randn(Bt, S, H, generator=g)                  # the caller's [Bt, S, H] order, read through strides
    whh = ((torch.rand(4 * H, H, generator=g) * 2 - 1) * (6.0 / (5 * H)) ** 0.5).to(torch.bfloat16)
    return [t.to(DEV) for t in (gates.reshape(S, Bt, 4 * H).contiguous(), c_all, dout, whh)]


def _bwd(inputs, S, Bt, H, drop_p):
    from vqa_attention_networks_b200 import ops
    gates, c_all, dout, whh = inputs
    dg = ops._sentinel_bf16((S * Bt, 4 * H), DEV)
    ops._call("vqa_b200_lstm_bwd", "lstm_bwd", ops._p(gates), ops._p(c_all), ops._p(dout), dout.stride(1),
              dout.stride(0), ops._p(whh), 1, ops._p(dg), S, Bt, H, float(drop_p), SEED, None, ops._st())
    torch.cuda.synchronize()
    return dg.view(torch.int16).view(S, Bt, 4 * H)


@pytest.mark.parametrize("H", [128, 256, 512, 1024])
@pytest.mark.parametrize("Bt", [1, 2, 7, 13, 26, 32])
@pytest.mark.parametrize("S", [1, 2, 256])
@pytest.mark.parametrize("drop_p", [0.0, 0.3])
def test_backward_row_split_dgates_bit_equal(H, Bt, S, drop_p):
    from vqa_attention_networks_b200 import ops
    gates, c_all, dout, whh = _inputs(S, Bt, H, 10 * H + Bt + S)
    n = max(Bt, 2)
    if Bt == 1:                                       # a single row runs in a batch of two copies, one in each half
        gates, c_all, dout = gates.repeat(1, 2, 1), c_all.repeat(1, 2, 1), dout.repeat(2, 1, 1)
    got = _bwd((gates, c_all, dout, whh), S, n, H, drop_p)
    assert not (got == -1).any()                      # every step published
    # The dropout mask hashes the time-major row t * Bt + b, so a row run alone would draw another mask: it gets the
    # batch's mask applied to its dout instead (the kernel multiplies by exactly these fp32 values, and drops to +0)
    # and runs with p = 0.
    mask = ops.dropout_mask(S * n, H, drop_p, SEED, DEV).view(S, n, H) if drop_p else torch.ones(S, n, H, device=DEV)
    for b in range(n):
        masked = torch.where(mask[:, b] > 0, dout[b] * mask[:, b], 0.0).unsqueeze(0)
        alone = (gates[:, b:b + 1].contiguous(), c_all[:, b:b + 1].contiguous(), masked, whh)
        assert torch.equal(got[:, b:b + 1], _bwd(alone, S, 1, H, 0.0)), b


def test_backward_clusters_setting_is_checked():
    inputs = _inputs(2, 3, 128, 0)
    os.environ["VQA_B200_LSTM_CLUSTERS"] = "2"        # read by the library at every launch
    try:
        with pytest.raises(RuntimeError, match="VQA_B200_LSTM_CLUSTERS"):
            _bwd(inputs, 2, 3, 128, 0.0)
    finally:
        os.environ.pop("VQA_B200_LSTM_CLUSTERS", None)
