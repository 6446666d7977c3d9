"""GPU parity of the persistent question-encoder recurrence (ops.LstmFn, csrc/lstm.cu) against the fp64 oracle
restatement of nn.LSTM (oracle.lstm_batch_first, pinned by the mhbcoatt golden fixtures) on the same seeded inputs.

The op computes with bf16 operands and fp32 accumulation / cell state (it is only used in bf16 mode), so the bound is
north_star's bf16 tolerance: relative L2 error <= 2e-2 on outputs; gradients <= 5e-2 (no singular op in the LSTM).
"""
import re

import pytest
import torch

from oracle import oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def _case(Bt, S, E, H, seed, xavier):
    g = torch.Generator().manual_seed(seed)
    bound = (6.0 / (4 * H + E)) ** 0.5 if xavier else H ** -0.5
    bound_h = (6.0 / (5 * H)) ** 0.5 if xavier else H ** -0.5
    W_ih = (torch.rand(4 * H, E, generator=g) * 2 - 1) * bound
    W_hh = (torch.rand(4 * H, H, generator=g) * 2 - 1) * bound_h
    b_ih = (torch.rand(4 * H, generator=g) * 2 - 1) * H ** -0.5
    b_hh = (torch.rand(4 * H, generator=g) * 2 - 1) * H ** -0.5
    # the reference's feed: tanh(embedding) stored [S, Bt, E], viewed batch_first as [Bt, S, E]
    x = torch.tanh(torch.randn(S, Bt, E, generator=g)).permute(1, 0, 2)
    cot = torch.randn(Bt, S, H, generator=g)
    return x, (W_ih, W_hh, b_ih, b_hh), cot


@pytest.mark.parametrize("Bt,S,E,H,xavier", [
    (3, 5, 20, 128, False),
    (32, 7, 64, 256, False),
    (17, 33, 300, 512, True),
    (26, 256, 300, 1024, True),          # BASELINE configs[1]: 256 steps over 26 rows, 300-d embeddings, H = 1024
    (26, 64, 600, 1024, False),          # glove feed (2 x 300), default nn.LSTM init
])
def test_lstm_matches_oracle(Bt, S, E, H, xavier):
    from vqa_attention_networks_b200 import ops
    assert ops.lstm_supported(Bt, H)
    x, params, cot = _case(Bt, S, E, H, 1000 + Bt + S, xavier)
    # oracle, fp64
    xo = x.double().requires_grad_(True)
    po = [p.double().requires_grad_(True) for p in params]
    ref = O.lstm_batch_first(xo, *po)
    (ref * cot.double()).sum().backward()
    # CUDA path
    xg = x.to(DEV).requires_grad_(True)
    pg = [p.to(DEV).requires_grad_(True) for p in params]
    out = ops.LstmFn.apply(xg, *pg, ops.WeightCache())
    assert out.shape == (Bt, S, H)
    (out * cot.to(DEV)).sum().backward()
    torch.cuda.synchronize()
    assert _rel(out, ref) <= 2e-2, _rel(out, ref)
    errs = {"dx": _rel(xg.grad, xo.grad)}
    for name, a, b in zip(("dW_ih", "dW_hh", "db_ih", "db_hh"), pg, po):
        errs[name] = _rel(a.grad, b.grad)
    assert max(errs.values()) <= 5e-2, errs
    # inference (no autograd state saved) gives the same outputs
    with torch.no_grad():
        out2 = ops.LstmFn.apply(x.to(DEV), *[p.detach() for p in pg], ops.WeightCache())
    assert torch.equal(out2, out.detach())


@pytest.mark.parametrize("Bt,S,E,H", [(5, 6, 24, 128), (20, 9, 40, 256), (32, 17, 64, 512), (26, 48, 300, 1024),
                                      (1, 200, 300, 1024), (2, 200, 300, 1024)])
def test_lstm_backward_variants_agree(Bt, S, E, H, monkeypatch):
    """The recurrence has a cluster form per direction (the default) and a cluster-free pair (VQA_B200_LSTM_CLUSTERS=0,
    also what runs when the clusters cannot all be co-resident): both must produce the same gradients."""
    from vqa_attention_networks_b200 import ops
    x, params, cot = _case(Bt, S, E, H, 77, True)
    xo = x.double().requires_grad_(True)
    po = [p.double().requires_grad_(True) for p in params]
    (O.lstm_batch_first(xo, *po) * cot.double()).sum().backward()
    grads = {}
    for clusters in ("1", "0"):
        monkeypatch.setenv("VQA_B200_LSTM_CLUSTERS", clusters)      # read by the library at every launch
        xg = x.to(DEV).requires_grad_(True)
        pg = [p.to(DEV).requires_grad_(True) for p in params]
        out = ops.LstmFn.apply(xg, *pg, ops.WeightCache())
        (out * cot.to(DEV)).sum().backward()
        torch.cuda.synchronize()
        grads[clusters] = [xg.grad] + [p.grad for p in pg]
        for a, b in zip(grads[clusters], [xo.grad] + [p.grad for p in po]):
            assert _rel(a, b) <= 5e-2, (clusters, _rel(a, b))
    for a, b in zip(grads["1"], grads["0"]):      # same bf16 operands, different summation order only
        assert _rel(a, b) <= 1e-3, _rel(a, b)


def _launched_lstm_kernels(prof):
    names = set()
    for ev in prof.events():
        m = re.search(r"lstm_\w+_kernel<[^>]*>", ev.name)
        if m and ev.device_type == torch.autograd.DeviceType.CUDA:
            names.add(m.group(0).replace(" ", ""))
    return names


@pytest.mark.parametrize("H", [128, 256, 512, 1024])
@pytest.mark.parametrize("Bt", [1, 26])
@pytest.mark.parametrize("clusters", [None, "0"])
def test_lstm_launch_forms(H, Bt, clusters, monkeypatch):
    """The kernels each form runs: by default the multicast forward in clusters of 4 and the row-split backward, with
    VQA_B200_LSTM_CLUSTERS=0 the sweep forward and the single-CTA backward.  A silent fallback would make the agreement
    tests compare a form with itself."""
    from torch.profiler import ProfilerActivity, profile
    from vqa_attention_networks_b200 import ops
    if clusters is None:
        monkeypatch.delenv("VQA_B200_LSTM_CLUSTERS", raising=False)
    else:
        monkeypatch.setenv("VQA_B200_LSTM_CLUSTERS", clusters)
    x, params, cot = _case(Bt, 4, 24, H, 6, True)
    xg = x.to(DEV).requires_grad_(True)
    pg = [p.to(DEV).requires_grad_(True) for p in params]
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ops.LstmFn.apply(xg, *pg, ops.WeightCache()).backward(cot.to(DEV))
        torch.cuda.synchronize()
    ks = H // 128
    if clusters is None:
        expected = {"lstm_fwd_kernel<%d,4>" % ks, "lstm_bwd_rows_kernel<%d>" % ks}
    else:
        expected = {"lstm_fwd_kernel<%d,1>" % ks, "lstm_bwd_kernel<%d>" % ks}
    assert _launched_lstm_kernels(prof) == expected


def test_lstm_rejects_unsupported_shapes():
    from vqa_attention_networks_b200 import ops
    assert not ops.lstm_supported(256, 1024)       # MFB's proper batch_first feed (256 rows per step): ops.LstmStepFn
    assert ops.lstm_steps_supported(256, 1024) and not ops.lstm_steps_supported(26, 1024)
    assert not ops.lstm_supported(26, 8)
    x = torch.zeros(40, 4, 16, device=DEV)
    W_ih, W_hh = torch.zeros(512, 16, device=DEV), torch.zeros(512, 128, device=DEV)
    b = torch.zeros(512, device=DEV)
    with pytest.raises(RuntimeError, match="lstm_fwd"):
        ops.LstmFn.apply(x, W_ih, W_hh, b, b, ops.WeightCache())


def test_mhbcoatt_fast_and_stock_lstm_agree(monkeypatch):
    """The drop-in module gives the same question states through the persistent kernel and through the stock
    nn.LSTM with the same parameters (bf16 tolerance), forward and parameter gradients."""
    import types
    from vqa_attention_networks_b200 import MHBCoAtt
    cfg = types.SimpleNamespace(model_name="mhb_coAtt", q_vocab_size=500, emb_dim=300, hidden_dim=1024, num_layers=1,
                                img_feature_channel=2048, img_feature_dim=196, a_vocab_size=100, glove=False)
    torch.manual_seed(3)
    model = MHBCoAtt(cfg).to(DEV).train()
    model.dropout_l.p = 0.0
    q = torch.randint(0, 500, (48, 26), device=DEV)
    cot = torch.randn(48, 26, 1024, device=DEV)
    res = {}
    for kind in ("fast", "stock"):
        monkeypatch.setenv("VQA_B200_LSTM", kind)
        model.zero_grad(set_to_none=True)
        f = model.question_features(q)
        (f * cot).sum().backward()
        res[kind] = (f.detach().clone(), {n: p.grad.clone() for n, p in model.named_parameters() if p.grad is not None})
    assert _rel(res["fast"][0], res["stock"][0]) <= 2e-2
    assert set(res["fast"][1]) == set(res["stock"][1])
    for n in res["stock"][1]:
        assert _rel(res["fast"][1][n], res["stock"][1][n]) <= 5e-2, n


@pytest.mark.parametrize("Bt,S,E,H,xavier", [
    (33, 4, 24, 128, False),             # just past the persistent kernels' 32 rows; ragged M tile
    (64, 26, 300, 1024, True),           # BASELINE configs[0]: MFB, batch 64, 26 tokens
    (200, 9, 300, 512, False),
    (512, 26, 300, 1024, True),          # BASELINE configs[3]: MFB-multilayer, 512 per GPU
])
def test_lstm_wide_batch_matches_oracle(Bt, S, E, H, xavier):
    """ops.LstmStepFn (mfb.py:68-70: T steps over N rows; per-step tcgen05 GEMM + cell kernels) against the fp64 oracle:
    same bounds as the persistent form."""
    from vqa_attention_networks_b200 import ops
    assert not ops.lstm_supported(Bt, H) and ops.lstm_steps_supported(Bt, H)
    x, params, cot = _case(Bt, S, E, H, 2000 + Bt + S, xavier)
    x = x.contiguous()                                 # MFB's feed is a plain [N, T, E] tensor
    xo = x.double().requires_grad_(True)
    po = [p.double().requires_grad_(True) for p in params]
    ref = O.lstm_batch_first(xo, *po)
    (ref * cot.double()).sum().backward()
    xg = x.to(DEV).requires_grad_(True)
    pg = [p.to(DEV).requires_grad_(True) for p in params]
    out = ops.LstmStepFn.apply(xg, *pg, ops.WeightCache())
    assert out.shape == (Bt, S, H) and out.is_contiguous()
    (out * cot.to(DEV)).sum().backward()
    torch.cuda.synchronize()
    assert _rel(out, ref) <= 2e-2, _rel(out, ref)
    errs = {"dx": _rel(xg.grad, xo.grad)}
    for name, a, b in zip(("dW_ih", "dW_hh", "db_ih", "db_hh"), pg, po):
        errs[name] = _rel(a.grad, b.grad)
    assert max(errs.values()) <= 5e-2, errs
    # inference (two rolling cell-state buffers, gates not saved, forward GEMMs not split along K): the same outputs up to
    # the summation order of the training pass's split-K accumulation, and bit-identical from run to run
    with torch.no_grad():
        out2 = ops.LstmStepFn.apply(x.to(DEV), *[p.detach() for p in pg], ops.WeightCache())
        out3 = ops.LstmStepFn.apply(x.to(DEV), *[p.detach() for p in pg], ops.WeightCache())
    assert _rel(out2, out) <= 1e-3
    assert torch.equal(out2, out3)


def test_lstm_wide_batch_strided_cotangent():
    """dL/dh arrives through its strides (a [Bt, S, H] view of a time-major tensor here): no transposing copy, same
    gradients as with a contiguous cotangent."""
    from vqa_attention_networks_b200 import ops
    Bt, S, E, H = 48, 6, 32, 256
    x, params, cot = _case(Bt, S, E, H, 5, False)
    res = []
    for strided in (False, True):
        xg = x.to(DEV).contiguous().requires_grad_(True)
        pg = [p.to(DEV).requires_grad_(True) for p in params]
        out = ops.LstmStepFn.apply(xg, *pg, ops.WeightCache())
        c = cot.to(DEV)
        if strided:
            c = c.permute(1, 0, 2).contiguous().permute(1, 0, 2)
            assert not c.is_contiguous()
        out.backward(c)
        res.append([xg.grad] + [p.grad for p in pg])
    for a, b in zip(*res):
        assert _rel(a, b) <= 1e-3


def test_mfb_fast_and_stock_lstm_agree(monkeypatch):
    """MFB's question encoder (mfb.py:68-70) through ops.run_lstm and through the stock nn.LSTM with the same
    parameters: question states and parameter gradients (bf16 tolerance)."""
    import types
    from vqa_attention_networks_b200 import MFB
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    cfg = types.SimpleNamespace(model_name="mfb", q_vocab_size=500, emb_dim=300, hidden_dim=1024, num_layers=1,
                                img_feature_channel=2048, img_feature_dim=196, a_vocab_size=100, glove=False)
    torch.manual_seed(3)
    model = MFB(cfg).to(DEV).train()
    model.dropout_l.p = 0.0
    q = torch.randint(0, 500, (64, 26), device=DEV)
    cot = torch.randn(64, 26, 1024, device=DEV)
    res = {}
    for kind in ("fast", "stock"):
        monkeypatch.setenv("VQA_B200_LSTM", kind)
        model.zero_grad(set_to_none=True)
        f = model.question_features(q)
        (f * cot).sum().backward()
        res[kind] = (f.detach().clone(), {n: p.grad.clone() for n, p in model.named_parameters() if p.grad is not None})
    assert _rel(res["fast"][0], res["stock"][0]) <= 2e-2
    assert set(res["fast"][1]) == set(res["stock"][1])
    for n in res["stock"][1]:
        assert _rel(res["fast"][1][n], res["stock"][1][n]) <= 5e-2, n


@pytest.mark.parametrize("form,Bt,S,E,H", [("persistent", 26, 40, 300, 1024), ("persistent", 7, 9, 24, 128),
                                           ("steps", 64, 26, 300, 1024), ("steps", 40, 5, 24, 256)])
@pytest.mark.parametrize("salted", [False, True])
def test_lstm_fused_output_dropout_is_the_mask(form, Bt, S, E, H, salted):
    """The dropout that follows the LSTM in the reference (mhb_coAtt.py:74, mfb.py:70) runs inside the recurrence
    kernels: the result is the clean output times the counter-hash mask of the time-major [S * Bt, H] matrix
    (ops.dropout_mask with the same seed / device salt), and the backward equals the clean backward of the masked
    cotangent."""
    from vqa_attention_networks_b200 import ops
    Fn = ops.LstmFn if form == "persistent" else ops.LstmStepFn
    x, params, cot = _case(Bt, S, E, H, 31, True)
    p, seed = 0.3, 90210
    salt = torch.tensor([5], dtype=torch.int64, device=DEV) if salted else None
    res = {}
    for kind in ("clean", "fused"):
        xg = x.to(DEV).contiguous().requires_grad_(True)
        pg = [q.to(DEV).requires_grad_(True) for q in params]
        cache = ops.WeightCache()
        if kind == "clean":
            out = Fn.apply(xg, *pg, cache)
        else:
            out = Fn.apply(xg, *pg, cache, p, seed, salt)
        res[kind] = (out, xg, pg)
    mask = ops.dropout_mask(S * Bt, H, p, seed, DEV, seed_dev=salt).view(S, Bt, H).permute(1, 0, 2)
    assert 0.6 < float((mask > 0).float().mean()) < 0.8
    if form == "persistent":
        assert torch.equal(res["fused"][0], res["clean"][0] * mask)
    else:                                                # training-mode step GEMMs are split along K: summation order
        assert _rel(res["fused"][0], res["clean"][0] * mask) <= 1e-3
        kept = mask > 0
        assert bool((res["fused"][0][~kept] == 0).all())
    c = cot.to(DEV)
    res["clean"][0].backward(c * mask)
    res["fused"][0].backward(c)
    for a, b in zip([res["fused"][1]] + res["fused"][2], [res["clean"][1]] + res["clean"][2]):
        assert _rel(a.grad, b.grad) <= 2e-3              # same inputs to the same kernels; split-K order in the GEMMs


def test_module_lstm_dropout_runs_in_the_kernel(monkeypatch):
    """MHBCoAtt / MFB in train mode: `dropout_l` is applied by the recurrence kernels (seed in last_lstm_drop_seed);
    VQA_B200_LSTM=stock and eval mode go through the stock modules."""
    import types
    from vqa_attention_networks_b200 import MHBCoAtt, MFB, ops
    for cls, name, N in ((MHBCoAtt, "mhb_coAtt", 12), (MFB, "mfb", 40)):
        cfg = types.SimpleNamespace(model_name=name, q_vocab_size=300, emb_dim=300, hidden_dim=1024, num_layers=1,
                                    img_feature_channel=2048, img_feature_dim=196, a_vocab_size=50, glove=False)
        torch.manual_seed(4)
        model = cls(cfg).to(DEV).train()
        q = torch.randint(0, 300, (N, 26), device=DEV)
        f = model.question_features(q)
        seed = model.last_lstm_drop_seed
        assert seed is not None
        model.dropout_l.p = 0.0
        clean = model.question_features(q)
        assert model.last_lstm_drop_seed is None
        model.dropout_l.p = 0.3
        # mask rows are time-major: MHBCoAtt's recurrence runs over the batch axis (S = N, Bt = T), MFB's over the tokens
        S, Bt = (N, 26) if cls is MHBCoAtt else (26, N)
        mask = ops.dropout_mask(S * Bt, 1024, 0.3, seed, DEV).view(S, Bt, 1024)
        mask = mask if cls is MHBCoAtt else mask.permute(1, 0, 2)
        assert _rel(f, clean * mask) <= 1e-4          # MFB at N = 40: training-mode step GEMMs are split along K
        assert bool((f[mask == 0] == 0).all())
        monkeypatch.setenv("VQA_B200_LSTM", "stock")
        model.question_features(q)
        assert model.last_lstm_drop_seed is None
        monkeypatch.delenv("VQA_B200_LSTM")
        model.eval()
        with torch.no_grad():
            e1, e2 = model.question_features(q), model.question_features(q)
        assert model.last_lstm_drop_seed is None and torch.equal(e1, e2)
