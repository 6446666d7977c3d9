"""The forward recurrence (csrc/lstm.cu, lstm_fwd_kernel) has two exchange forms for h_{t-1}: one TMA load per cluster
of 4 CTAs multicast to its CTAs (the default), and every CTA sweeping its slices out of L2 (VQA_B200_LSTM_CLUSTERS=0,
also the fallback when the clusters cannot all be co-resident).  Only the data movement differs -- same operands, same
MMA and reduction order -- so every result must be bit-identical: the outputs (with and without the fused output
dropout), the saved activated gates, the cell states and the bf16 exchange buffer the dW_hh gradient reads."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _run(gates0, whh, S, Bt, H, drop_p, train, clusters):
    from vqa_attention_networks_b200 import ops
    gates = gates0.clone()
    out = torch.empty((S, Bt, H), device=DEV, dtype=torch.float32)
    hb = ops._sentinel_bf16((S + 1, Bt, H), DEV)
    hb[0].zero_()
    c_all = torch.empty((S, Bt, H), device=DEV, dtype=torch.float32) if train else None
    try:
        if clusters is None:                        # read by the library at every launch
            os.environ.pop("VQA_B200_LSTM_CLUSTERS", None)
        else:
            os.environ["VQA_B200_LSTM_CLUSTERS"] = clusters
        ops._call("vqa_b200_lstm_fwd", "lstm_fwd", ops._p(gates), ops._p(whh), ops._p(out), ops._p(hb), ops._p(c_all),
                  S, Bt, H, float(drop_p), 1234, None, ops._st())
        torch.cuda.synchronize()
    finally:
        os.environ.pop("VQA_B200_LSTM_CLUSTERS", None)
    res = {"out": out, "hb": hb.view(torch.int16)}
    if train:
        res["gates"] = gates
        res["c_all"] = c_all
    return res


def _inputs(S, Bt, H, seed):
    g = torch.Generator().manual_seed(seed)
    gates = (torch.randn(S, Bt, 4 * H, generator=g) * 0.5).to(DEV)
    whh = ((torch.rand(4 * H, H, generator=g) * 2 - 1) * (6.0 / (5 * H)) ** 0.5).to(DEV).to(torch.bfloat16)
    return gates, whh


def _assert_forms_equal(S, Bt, H, drop_p, train, seed):
    gates, whh = _inputs(S, Bt, H, seed)
    ref = _run(gates, whh, S, Bt, H, drop_p, train, "0")
    assert not (ref["hb"] == -1).any()             # every step published
    got = _run(gates, whh, S, Bt, H, drop_p, train, None)
    for k in ref:
        assert torch.equal(got[k], ref[k]), k


@pytest.mark.parametrize("H", [128, 256, 512, 1024])
@pytest.mark.parametrize("Bt", [1, 7, 26, 32])
@pytest.mark.parametrize("S", [1, 2, 256])
@pytest.mark.parametrize("drop_p", [0.0, 0.3])
def test_forward_exchange_forms_bit_equal(H, Bt, S, drop_p):
    _assert_forms_equal(S, Bt, H, drop_p, True, 10 * H + Bt + S)


def test_forward_exchange_forms_bit_equal_long_inference():
    """The inference form of the c5 question encoder: 4096 steps over 26 rows, no saved states."""
    _assert_forms_equal(4096, 26, 1024, 0.0, False, 5)


def test_forward_clusters_setting_is_checked():
    gates, whh = _inputs(2, 3, 128, 0)
    with pytest.raises(RuntimeError, match="VQA_B200_LSTM_CLUSTERS"):
        _run(gates, whh, 2, 3, 128, 0.0, True, "bogus")
