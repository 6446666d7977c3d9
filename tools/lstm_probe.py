"""Times the persistent recurrence (ops.LstmFn) on config 2's shape -- 256 steps over 26 rows, 300 -> 1024 -- forward
(training form: gates and cell states saved) and backward, CUDA events over 20 calls; the forward is also
checked for run-to-run bit equality; each forward exchange form (sweep / multicast) in turn.  (Used for the A/B runs of round 2: 16-byte publications -45 us forward / -36 us
backward; speculative sweeps without the canary spin +13 %; one barrier per step with double-buffered partial tiles
+13 %; poll backoff +7 %.)"""
import json, os, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vqa_attention_networks_b200 import ops

dev = "cuda:0"
Bt, S, E, H = 26, int(os.environ.get("S", 256)), 300, 1024
g = torch.Generator().manual_seed(0)
x = torch.tanh(torch.randn(S, Bt, E, generator=g)).permute(1, 0, 2).to(dev).requires_grad_(True)
W_ih = ((torch.rand(4 * H, E, generator=g) * 2 - 1) * (6.0 / (4 * H + E)) ** 0.5).to(dev).requires_grad_(True)
W_hh = ((torch.rand(4 * H, H, generator=g) * 2 - 1) * (6.0 / (5 * H)) ** 0.5).to(dev).requires_grad_(True)
b = ((torch.rand(4 * H, generator=g) * 2 - 1) * H ** -0.5).to(dev).requires_grad_(True)
cot = torch.randn(Bt, S, H, generator=g).to(dev)
cache = ops.WeightCache()


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


def fwd_bwd():
    for t in (x, W_ih, W_hh, b):
        t.grad = None
    ops.LstmFn.apply(x, W_ih, W_hh, b, b, cache).backward(cot)


# A/B of the forward exchange (VQA_B200_LSTM_EXCHANGE, read by the library at every launch), alternated twice
res, ref = {}, None
for rep in range(2):
    for mode in ("sweep", "multicast"):
        os.environ["VQA_B200_LSTM_EXCHANGE"] = mode
        with torch.no_grad():
            out = ops.LstmFn.apply(x.detach(), W_ih.detach(), W_hh.detach(), b.detach(), b.detach(), cache)
            t_inf = timed(lambda: ops.LstmFn.apply(x.detach(), W_ih.detach(), W_hh.detach(), b.detach(), b.detach(), cache))
        t_fwd = timed(lambda: ops.LstmFn.apply(x, W_ih, W_hh, b, b, cache))
        if ref is None:
            ref = out.clone()
        same = bool(torch.equal(out, ref))
        r = {"fwd_inference_ms": round(t_inf, 4), "fwd_training_ms": round(t_fwd, 4), "bit_equal_to_first_run": same,
             "fwd_bwd_ms": round(timed(fwd_bwd), 4)}
        res["%s_%d" % (mode, rep)] = r
        print(mode, rep, r, flush=True)
os.environ.pop("VQA_B200_LSTM_EXCHANGE", None)
os.makedirs("gpurun_out", exist_ok=True)
json.dump(res, open("gpurun_out/lstm_probe.json", "w"), indent=1)
