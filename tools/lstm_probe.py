"""Times the persistent recurrence on config 2's shape -- 256 steps over 26 rows, 300 -> 1024 -- CUDA events over 20
calls: the backward kernel alone (vqa_b200_lstm_bwd on saved activations, a fresh sentinel-filled dg per call), and
ops.LstmFn forward (training and inference form) plus fwd+bwd; the outputs and the backward's dg are also checked for
bit equality against the first form.  S and Bt can be overridden from the environment (S=..., Bt=...).

The A/B subject is one library switch, read at every launch, alternated twice in one process:
AB="VARIABLE=value1,value2" (default VQA_B200_LSTM_CLUSTERS=0,1: the cluster-free forms against the cluster forms,
whose backward dg differ from theirs in summation order).
(Earlier A/B runs with it, round 2: 16-byte publications -45 us forward / -36 us backward; speculative sweeps without the
canary spin +13 %; one barrier per step with double-buffered partial tiles +13 %; poll backoff +7 %.)

    python tools/lstm_probe.py [out.json]        (without a path the JSON goes to stdout only)"""
import json, os, subprocess, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vqa_attention_networks_b200 import ops

dev = "cuda:0"
Bt, S, E, H = int(os.environ.get("Bt", 26)), int(os.environ.get("S", 256)), 300, 1024
var, vals = os.environ.get("AB", "VQA_B200_LSTM_CLUSTERS=0,1").split("=")
vals = vals.split(",")
g = torch.Generator().manual_seed(0)
x = torch.tanh(torch.randn(S, Bt, E, generator=g)).permute(1, 0, 2).to(dev).requires_grad_(True)
W_ih = ((torch.rand(4 * H, E, generator=g) * 2 - 1) * (6.0 / (4 * H + E)) ** 0.5).to(dev).requires_grad_(True)
W_hh = ((torch.rand(4 * H, H, generator=g) * 2 - 1) * (6.0 / (5 * H)) ** 0.5).to(dev).requires_grad_(True)
b = ((torch.rand(4 * H, generator=g) * 2 - 1) * H ** -0.5).to(dev).requires_grad_(True)
cot = torch.randn(Bt, S, H, generator=g).to(dev)
cache = ops.WeightCache()

# inputs of the backward kernel alone: activated gates and cell states saved by one training-form forward
whh = W_hh.detach().to(torch.bfloat16).contiguous()
gates = (torch.randn(S, Bt, 4 * H, generator=g) * 0.5).to(dev)
c_all = torch.empty((S, Bt, H), device=dev)
hb = ops._sentinel_bf16((S + 1, Bt, H), dev)
hb[0].zero_()
ops._call("vqa_b200_lstm_fwd", "lstm_fwd", ops._p(gates), ops._p(whh), ops._p(torch.empty_like(c_all)), ops._p(hb),
          ops._p(c_all), S, Bt, H, 0.0, 0, None, ops._st())


def timed(fn, n=20):
    for _ in range(3):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def bwd_kernel(n=20):
    """ms per call of the backward kernel alone; returns (ms, dg of the last call)."""
    dgs = [ops._sentinel_bf16((S * Bt, 4 * H), dev) for _ in range(n + 3)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i, dg in enumerate(dgs):
        if i == 3:
            torch.cuda.synchronize()
            e0.record()
        ops._call("vqa_b200_lstm_bwd", "lstm_bwd", ops._p(gates), ops._p(c_all), ops._p(cot), cot.stride(1),
                  cot.stride(0), ops._p(whh), 1, ops._p(dg), S, Bt, H, 0.0, 0, None, ops._st())
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n, dgs[-1]


def fwd_bwd():
    for t in (x, W_ih, W_hh, b):
        t.grad = None
    ops.LstmFn.apply(x, W_ih, W_hh, b, b, cache).backward(cot)


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return str(e)


res, ref = {"card": card(), "shape": {"S": S, "Bt": Bt, "E": E, "H": H}, "ab": var}, None
for rep in range(2):
    for v in vals:
        os.environ[var] = v
        t_bwd, dg = bwd_kernel()
        with torch.no_grad():
            out = ops.LstmFn.apply(x.detach(), W_ih.detach(), W_hh.detach(), b.detach(), b.detach(), cache)
            t_inf = timed(lambda: ops.LstmFn.apply(x.detach(), W_ih.detach(), W_hh.detach(), b.detach(), b.detach(), cache))
        t_fwd = timed(lambda: ops.LstmFn.apply(x, W_ih, W_hh, b, b, cache))
        if ref is None:
            ref = (out.clone(), dg.clone())
        r = {"bwd_kernel_ms": round(t_bwd, 4), "fwd_inference_ms": round(t_inf, 4), "fwd_training_ms": round(t_fwd, 4),
             "fwd_bwd_ms": round(timed(fwd_bwd), 4),
             "out_bit_equal_to_first": bool(torch.equal(out, ref[0])),
             "dg_bit_equal_to_first": bool(torch.equal(dg.view(torch.int16), ref[1].view(torch.int16)))}
        res["%s_%d" % (v, rep)] = r
        print(var, v, rep, r, flush=True)
os.environ.pop(var, None)
print(json.dumps(res, indent=1))
if len(sys.argv) > 1:
    dst = sys.argv[1]
    if os.path.dirname(dst):
        os.makedirs(os.path.dirname(dst), exist_ok=True)
    with open(dst, "w") as f:
        json.dump(res, f, indent=1)
