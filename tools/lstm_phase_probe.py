"""Per-phase cycle counters of the recurrence kernels over ALL CTAs, on config 2's shape (S=256 steps over Bt=26 rows,
300 -> 1024), forward (training form) and backward, for the default cluster forms (`clusters`: multicast forward,
row-split backward) and the cluster-free pair (`cluster_free`: sweep forward, single-CTA backward), chosen through
VQA_B200_LSTM_CLUSTERS.

Builds the library with VQA_B200_DEBUG=1 (instrumented kernels + the vqa_b200_debug_set_lstm hook) into a temporary
copy of the package, so the tree's release library is left alone.  Thread 0 of every CTA accumulates clock64() deltas
per phase over the whole sequence; the JSON holds, per phase, the median and the max over CTAs in SM cycles per step
and the share of the step, plus the card's name and power limit.

    python tools/lstm_phase_probe.py [out.json]        (without a path the JSON goes to stdout only)
"""
import json
import os
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FWD_PHASES = ["spin", "exchange_and_mma", "partial_store", "cta_barrier", "gate_math_publish", "stores",
              "end_barrier"]
BWD_PHASES = ["spin", "exchange_and_mma", "partial_store", "cta_reduce", "cluster_barrier_gate_math_publish"]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": plim, "max_sm_clock": clk}
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}


def build_debug_copy():
    tmp = tempfile.mkdtemp(prefix="vqa_lstm_phase_probe_")
    shutil.copytree(os.path.join(ROOT, "vqa_attention_networks_b200"), os.path.join(tmp, "vqa_attention_networks_b200"),
                    ignore=shutil.ignore_patterns("*.so", "build", "__pycache__", ".build.lock", "*.tmp"))
    shutil.copytree(os.path.join(ROOT, "include"), os.path.join(tmp, "include"))
    os.environ["VQA_B200_DEBUG"] = "1"
    sys.path.insert(0, tmp)
    from vqa_attention_networks_b200 import build
    assert os.path.dirname(build.__file__).startswith(tmp), build.__file__
    build.build(force=True)
    return tmp


def summarise(rows, names, steps):
    import numpy as np
    out = {}
    tot = rows[:, :len(names)].sum(axis=1)
    for i, n in enumerate(names):
        v = rows[:, i] / steps
        out[n] = {"median_cycles_per_step": round(float(np.median(v)), 1), "max_cycles_per_step": round(float(v.max()), 1),
                  "median_share": round(float(np.median(rows[:, i] / np.maximum(tot, 1))), 4)}
    out["total"] = {"median_cycles_per_step": round(float(np.median(tot / steps)), 1),
                    "min_cycles_per_step": round(float(tot.min() / steps), 1),
                    "max_cycles_per_step": round(float(tot.max() / steps), 1)}
    out["retries"] = {"median": float(np.median(rows[:, 7])), "max": int(rows[:, 7].max()),
                      "sum": int(rows[:, 7].sum())}
    return out


def main():
    dst = sys.argv[1] if len(sys.argv) > 1 else None
    tmp = build_debug_copy()
    try:
        import torch
        from vqa_attention_networks_b200 import _lib, ops
        L = _lib.load()
        assert hasattr(L, "vqa_b200_debug_set_lstm"), "debug hook missing: not a VQA_B200_DEBUG build"
        dev = "cuda:0"
        Bt, S, E, H = 26, 256, 300, 1024
        ncta = H // 8
        g = torch.Generator().manual_seed(0)
        x = torch.tanh(torch.randn(S, Bt, E, generator=g)).permute(1, 0, 2).to(dev).requires_grad_(True)
        W_ih = ((torch.rand(4 * H, E, generator=g) * 2 - 1) * (6.0 / (4 * H + E)) ** 0.5).to(dev).requires_grad_(True)
        W_hh = ((torch.rand(4 * H, H, generator=g) * 2 - 1) * (6.0 / (5 * H)) ** 0.5).to(dev).requires_grad_(True)
        b = ((torch.rand(4 * H, generator=g) * 2 - 1) * H ** -0.5).to(dev).requires_grad_(True)
        cot = torch.randn(Bt, S, H, generator=g).to(dev)
        cache = ops.WeightCache()
        dbg = torch.zeros(ncta * 16, dtype=torch.int64, device=dev)
        res = {"card": card(), "shape": {"S": S, "Bt": Bt, "E": E, "H": H}, "unit": "SM cycles (clock64)",
               "note": "thread 0 of every CTA; forward and backward of the last of 5 fwd+bwd calls"}
        for mode, clusters in (("clusters", "1"), ("cluster_free", "0")):
            os.environ["VQA_B200_LSTM_CLUSTERS"] = clusters
            L.vqa_b200_debug_set_lstm(ctypes_ptr(dbg), ncta << 16)
            for _ in range(5):
                for t in (x, W_ih, W_hh, b):
                    t.grad = None
                ops.LstmFn.apply(x, W_ih, W_hh, b, b, cache).backward(cot)
            torch.cuda.synchronize()
            L.vqa_b200_debug_set_lstm(None, 0)
            os.environ.pop("VQA_B200_LSTM_CLUSTERS")
            rows = dbg.view(ncta, 16).cpu().numpy()
            res[mode] = {"forward": summarise(rows[:, :8], FWD_PHASES, S),
                         "backward": summarise(rows[:, 8:], BWD_PHASES, S - 1)}
            print(mode, json.dumps(res[mode]), flush=True)
        print(json.dumps(res, indent=1))
        if dst:
            d = os.path.dirname(dst)
            if d:
                os.makedirs(d, exist_ok=True)
            with open(dst, "w") as f:
                json.dump(res, f, indent=1)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def ctypes_ptr(t):
    import ctypes
    return ctypes.c_void_p(t.data_ptr())


if __name__ == "__main__":
    main()
