"""Run-to-run agreement of what `bench.py --dump-outputs` writes, and of the parameters it leaves out.

    python tools/dump_repro.py OUT.json [bench.py arguments ...]

Runs bench.py twice with the given arguments plus --dump-outputs and compares every dumped array.  For the train
configurations it then trains the same model from the same seed twice more, each time in a fresh process, for as many
eager steps as the bench's warm-up and timed steps together (max(3, W) + K), and compares every parameter.  Writes the
figures, the command and the card (name, power limit) to OUT.json.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def compare(a, b):
    a, b = a.astype(np.float64), b.astype(np.float64)
    d = np.abs(a - b)
    top = float(np.abs(a).max()) if a.size else 0.0
    return {"shape": list(a.shape), "max_abs": float(d.max()) if d.size else 0.0,
            "max_abs_over_max": float(d.max()) / max(top, 1e-30) if d.size else 0.0,
            "rel_l2": float(np.linalg.norm(a - b)) / max(float(np.linalg.norm(a)), 1e-30)}


def train_params(out, config, steps, precision, batch):
    """Eager train steps of a bench configuration (one process, cuda:0); saves every parameter to `out` (.npz)."""
    import torch
    sys.path.insert(0, ROOT)
    import bench
    from vqa_attention_networks_b200.optim import FusedAdam
    from vqa_attention_networks_b200.train import TrainStep
    wl = bench.WORKLOADS[config]
    dev = torch.device("cuda", 0)
    model = bench.build_model(torch, wl)
    model.precision = precision
    model = model.to(dev).train()
    opt = FusedAdam(model.parameters(), lr=wl["lr"]).attach(model)
    crit = torch.nn.KLDivLoss() if wl["target"] == "soft" else torch.nn.CrossEntropyLoss()
    step = TrainStep(model, crit, opt)
    data = [tuple(t.to(dev) for t in bench.synth_batch(torch, batch or wl["batch"], 1234 + i, L=wl["L"],
                                                       target=wl["target"])) for i in range(2)]
    for i in range(steps):
        step(*data[i % 2])
    torch.cuda.synchronize()
    np.savez(out, **{n: p.detach().float().cpu().numpy() for n, p in model.named_parameters()})


def main():
    if sys.argv[1] == "--train-params":
        out, config, steps, precision, batch = sys.argv[2:7]
        train_params(out, config, int(steps), precision, int(batch))
        return
    out, bench_args = sys.argv[1], sys.argv[2:]
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c2")
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--precision", default="bf16")
    ap.add_argument("--batch", type=int, default=0)
    known, _ = ap.parse_known_args(bench_args)
    sys.path.insert(0, ROOT)
    import bench
    wl = bench.WORKLOADS[known.config]
    card = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    res = {"command": "python tools/dump_repro.py %s" % " ".join(sys.argv[1:]), "card": card, "dump": {},
           "parameters": None}
    with tempfile.TemporaryDirectory() as tmp:
        dirs = [os.path.join(tmp, "dump%d" % r) for r in (1, 2)]
        for d in dirs:
            subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *bench_args, "--dump-outputs", d],
                           check=True, stdout=subprocess.DEVNULL)
        for f in sorted(os.listdir(dirs[0])):
            res["dump"][f[:-4]] = compare(np.load(os.path.join(dirs[0], f)), np.load(os.path.join(dirs[1], f)))
        if wl["target"] is not None:
            n = max(3, known.warmup) + known.steps
            paths = [os.path.join(tmp, "params%d.npz" % r) for r in (1, 2)]
            for p in paths:
                subprocess.run([sys.executable, os.path.abspath(__file__), "--train-params", p, known.config, str(n),
                                known.precision, str(known.batch)], check=True)
            a, b = np.load(paths[0]), np.load(paths[1])
            arrays = {k: compare(a[k], b[k]) for k in a.files}
            res["parameters"] = {"eager_steps": n, "arrays": arrays,
                                 "worst_max_abs": max(arrays.items(), key=lambda kv: kv[1]["max_abs"])[0]}
    json.dump(res, open(out, "w"), indent=1)
    print(json.dumps({"dump": res["dump"], "worst_parameter": res["parameters"] and
                      {res["parameters"]["worst_max_abs"]:
                       res["parameters"]["arrays"][res["parameters"]["worst_max_abs"]]}}))


if __name__ == "__main__":
    main()
