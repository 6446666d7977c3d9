"""bench.py -- the BASELINE.json configurations of the fusion / co-attention hot path on N B200s of one node.

    python bench.py [--config c1|c2|c3|c4|c5] [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--batch B] [--precision bf16|fp32] [--dump-outputs DIR]

Configurations (BASELINE.json `configs`, SURVEY.md 8d "Config -> concrete run"); the default, and the one the metric is
quoted on, is c2:
  c1  MFB('mfb') train step, batch 64 (CrossEntropyLoss + Adam, solver.py:26-30,68-94)
  c2  MHBCoAtt (MFH co-attention, 2 MFB blocks, 2 glimpses) train step, batch 256 per GPU (KLDivLoss + Adam)
  c3  HieCoAtten(196, 26, 2048, 15000, 512, 3000) train step, batch 256 per GPU (CrossEntropyLoss + Adam 1e-4,
      train_hfd.py:62-82)
  c4  MFB('mfb-multilayer') data-parallel train step, batch 512 per GPU, gradient all-reduce over NCCL
  c5  MHBCoAtt eval forward, 100-region bottom-up features, global batch swept 1..4096, batch-sharded over the GPUs
      with no communication (CUDA-graph replay per batch shape)
Synthetic 14x14x2048 (c5: 100x2048) relu(N(0,1)) features, 26-token questions, 15k vocab, 3000 answers.

Prints ONE JSON line (rank 0).  `value` = whole-job samples/s with inputs resident in HBM; `e2e` = the same step through
the public module API with HOST (pinned) inputs, H2D copies and a D2H read of the result inside the timed region;
`roofline` = the configuration's dominant kernel timed live with CUDA events; `cpu_baseline` = the oracle port of the
reference's algorithm on the host cores (bounded sample).  `--impl reference` times that CPU path alone (rank 0 only).

`--dump-outputs DIR` writes what the last timed step returned to its caller on rank 0 as DIR/<name>.npy (float32):
for c1..c4 the loss of rank 0's batch, for c5 the log-probabilities of rank 0's rows of the largest batch.  Inputs,
weights and dropout seeds depend on the arguments only, so two builds run with the same arguments can be compared array
by array.  The parameters are not dumped: they carry every step before the last, and Adam turns the rounding noise of
the atomic gradient sums into whole +-lr steps wherever a gradient is near zero, so they differ from run to run by far
more than rounding (tools/dump_repro.py measures both).

The tree may be read-only: scratch files (the feature shard, the clock samples) go to the temporary directory.
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import subprocess
import sys
import tempfile
import time
import types

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

L_REGIONS, D_FEAT, T_TOK, H_DIM, VOCAB, ANSWERS, E_HIE = 196, 2048, 26, 1024, 15000, 3000, 512
_OUT = sys.stdout

# model: which drop-in class; target: "soft" = [N, A] rows summing to 1 (KLDivLoss, solver.py:27), "hard" = int64 labels
WORKLOADS = {
    "c1": dict(model="mfb", name="mfb", batch=64, L=196, target="hard", lr=7e-4, metric="MFB co-attn train samples/s",
               what="MFB('mfb', k=5, o=1000, 2 degenerate glimpses) train step: fwd + CrossEntropyLoss + bwd + Adam"),
    "c2": dict(model="mhbcoatt", name="mhb_coAtt", batch=256, L=196, target="soft", lr=7e-4,
               metric="MFH co-attn train samples/s",
               what="MHBCoAtt (MFH co-attention, 2 MFB blocks, 2 glimpses) train step: fwd + KLDivLoss + bwd + Adam"),
    "c3": dict(model="hie", name="hieCoAtten", batch=256, L=196, target="hard", lr=1e-4,
               metric="HieCoAtten train samples/s",
               what="HieCoAtten(block 196, word 26, img 2048, vocab 15000, embed 512, out 3000) train step: fwd + "
                    "CrossEntropyLoss + bwd + Adam"),
    "c4": dict(model="mfb", name="mfb-multilayer", batch=512, L=196, target="hard", lr=7e-4,
               metric="MFB-multilayer data-parallel train samples/s",
               what="MFB('mfb-multilayer') data-parallel train step: fwd + CrossEntropyLoss + bwd + gradient all-reduce "
                    "+ Adam"),
    "c5": dict(model="mhbcoatt", name="mhb_coAtt", batch=4096, L=100, target=None, lr=0.0,
               metric="MFH inference samples/s",
               what="MHBCoAtt eval forward on 100-region bottom-up features, global batch sweep 1..4096, batch-sharded"),
}


def cfg_ns(L=L_REGIONS, name="mhb_coAtt"):
    return types.SimpleNamespace(model_name=name, q_vocab_size=VOCAB, emb_dim=300, hidden_dim=H_DIM, num_layers=1,
                                 img_feature_channel=D_FEAT, img_feature_dim=L, a_vocab_size=ANSWERS, glove=False)


def build_model(torch, wl, seed=0):
    """The drop-in module of a workload with the reference's own init recipe: train_models.py:54-56 (Xavier on every
    non-bias parameter) for the solver.py models, torch's defaults for HieCoAtten (train_hfd.py:62-66 has no init loop)."""
    import vqa_attention_networks_b200 as V
    torch.manual_seed(seed)
    if wl["model"] == "hie":
        return V.HieCoAtten(block_num=wl["L"], word_num=T_TOK, img_size=D_FEAT, vocab_size=VOCAB, embed_size=E_HIE,
                            output_size=ANSWERS)
    model = (V.MHBCoAtt if wl["model"] == "mhbcoatt" else V.MFB)(cfg_ns(wl["L"], wl["name"]))
    for n, p in model.named_parameters():
        if n.find("bias") == -1:
            torch.nn.init.xavier_uniform_(p)
    return model


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        try:
            d = json.load(open(path))
            return {"bf16_sustained": float(d["bf16_tflops_sustained"]), "bf16_burst": float(d["bf16_tflops"]),
                    "hbm": float(d["hbm_gbs"]), "source": "measured"}
        except Exception:
            pass
    return {"bf16_sustained": 1400.0, "bf16_burst": 1590.0, "hbm": 6650.0, "source": "fallback"}


DUMP_BYTES = 60 << 20        # payload of all --dump-outputs arrays together; the .npy headers fit in the rest of 64 MB


def dump_outputs(out_dir, arrays):
    """Write each tensor of `arrays` (name -> tensor) as <out_dir>/<name>.npy in float32.  A tensor larger than its equal
    share of DUMP_BYTES is written as a sample of its flattened elements, at positions drawn from a fixed seed (the same
    positions in every run)."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // 4 // len(arrays)
    for name, t in arrays.items():
        a = t.detach().float()
        how = "shape %s" % (list(a.shape),)
        if a.numel() > share:
            pos = np.sort(np.random.default_rng(0).choice(a.numel(), share, replace=False))
            a = a.reshape(-1)[torch.from_numpy(pos).to(a.device)]
            how += ", seeded sample of %d elements" % share
        np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy())
        print("bench: dumped %s (%s)" % (name, how), file=sys.stderr)


# ------------------------------------------------------------------------------------------------
# synthetic data (SURVEY.md 8d)
# ------------------------------------------------------------------------------------------------
def synth_batch(torch, n, seed, pin=False, L=L_REGIONS, target="soft"):
    g = torch.Generator().manual_seed(seed)
    img = torch.empty(n, L, D_FEAT)
    img.normal_(generator=g).relu_()
    q = torch.randint(0, VOCAB, (n, T_TOK), generator=g)
    if target == "hard":
        tgt = torch.randint(0, ANSWERS, (n,), generator=g)
    else:
        tgt = torch.zeros(n, ANSWERS)
        idx = torch.randint(0, ANSWERS, (n, 10), generator=g)
        w = torch.rand(n, 10, generator=g) + 0.1
        tgt.scatter_add_(1, idx, w)
        tgt /= tgt.sum(1, keepdim=True)
    if pin:
        img, q, tgt = img.pin_memory(), q.pin_memory(), tgt.pin_memory()
    return img, q, tgt


def h2d_bandwidth_gbs(torch, host_tensor, dev, reps=3):
    """Pinned host -> device copy rate of one feature batch (GB/s), measured with CUDA events."""
    dst = torch.empty_like(host_tensor, device=dev)
    dst.copy_(host_tensor, non_blocking=True)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        dst.copy_(host_tensor, non_blocking=True)
    e1.record()
    torch.cuda.synchronize()
    return host_tensor.numel() * host_tensor.element_size() * reps / (e0.elapsed_time(e1) * 1e-3) / 1e9


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 20 ms.  The process is started BEFORE the warm-up (nvidia-smi
    needs a few hundred ms to come up, longer than a short timed region); only samples whose timestamp falls inside the
    window marked by begin()/end() -- the timed region -- are used."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu = str(gpu_index)
        self.proc = None
        self.path = os.path.join(tempfile.gettempdir(), "vqa_b200_clocks_%d.csv" % os.getpid())
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", self.gpu, "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def begin(self):
        self.t0 = time.time()

    def end(self):
        self.t1 = time.time()

    def stop(self):
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons, allsm = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(parts[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                c, m = float(parts[1]), float(parts[2])
            except ValueError:
                continue
            allsm.append(c)
            if self.t0 is not None and self.t1 is not None and not (self.t0 - 0.02 <= ts <= self.t1 + 0.02):
                continue
            sm.append(c)
            mx.append(m)
            for nme, val in zip(names, parts[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(nme)
        if sm:
            sm.sort()
            out = {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}
        elif allsm:      # region shorter than the sampling period: fall back to everything sampled since the warm-up
            allsm.sort()
            out = {"sm_mhz": allsm[len(allsm) // 2], "sm_max_mhz": None, "reasons": [], "samples": 0,
                   "note": "no sample inside the timed window; median over warm-up + timed region"}
        try:
            os.remove(self.path)
        except OSError:
            pass
        return out


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's algorithm on the host cores (oracle port; the reference itself is Python
# under /root/reference, which does not exist on the GPU box)
# ------------------------------------------------------------------------------------------------
def cpu_reference_run(wl, steps, warmup, sample_batch, budget_s=240.0):
    """`steps` timed + `warmup` untimed steps of the oracle port of workload `wl` at batch `sample_batch`.  If the first
    step shows that the run would exceed `budget_s`, the sample is halved (once or more) before timing starts."""
    import torch
    import torch.nn.functional as F
    from oracle import oracle as O          # checker / baseline only (never on the product path)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    model = build_model(torch, wl)          # parameter container only (never called)
    params = {k: v.detach().clone().requires_grad_(v.is_floating_point()) for k, v in model.state_dict().items()}
    train = wl["target"] is not None
    opt = torch.optim.Adam([v for v in params.values() if v.requires_grad], lr=wl["lr"] or 1e-3) if train else None
    gen = torch.Generator().manual_seed(99)
    L = wl["L"]

    def m(shape, p):
        return (torch.rand(shape, generator=gen) >= p).float() / (1 - p)

    def forward(img, q, n):
        if wl["model"] == "mhbcoatt":
            masks = None
            if train:
                masks = {"l": m((T_TOK, n, H_DIM), 0.3), "m1": m((n, L, 5000), 0.1), "m2": m((n, 5000), 0.1),
                         "m3": m((n, 5000), 0.1)}
            return O.mhbcoatt_forward(params, img, q, None, masks)
        if wl["model"] == "mfb":
            masks = {"l": m((n, T_TOK, H_DIM), 0.3), "m2": m((n, 5000), 0.1)}
            return O.mfb_forward(params, img, q, wl["name"] == "mfb-multilayer", masks)
        masks = [m((n, L, E_HIE), 0.5), m((n, T_TOK, E_HIE), 0.5), m((n, T_TOK, L), 0.5), m((n, L, E_HIE), 0.5),
                 m((n, T_TOK, E_HIE), 0.5)]
        return O.hiecoatten_forward(params, img, q, masks)[0]

    def make(n):
        img, q, tgt = synth_batch(torch, n, 1234, L=L, target=wl["target"] or "soft")

        def step():
            if not train:
                with torch.no_grad():
                    return float(forward(img, q, n).argmax(1).sum())
            out = forward(img, q, n)
            loss = F.kl_div(out, tgt, reduction="mean") if wl["target"] == "soft" else F.cross_entropy(out, tgt)
            opt.zero_grad()
            loss.backward()
            opt.step()
            return float(loss)
        return step

    n = sample_batch
    while True:
        step = make(n)
        t0 = time.perf_counter()
        step()                               # first (untimed) step: also the probe for the time budget
        t1 = time.perf_counter() - t0
        if t1 * (steps + warmup) <= budget_s or n <= 4:
            break
        n = max(4, n // 2)
    for _ in range(max(0, warmup - 1)):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / max(1, steps)
    kind = "fwd+loss+bwd+Adam, train-mode dropout masks" if train else "eval forward under no_grad"
    return {"value": n / dt, "unit": "samples/s", "cores": cores, "kind": "port",
            "sample": "oracle port of %s (%s), batch %d x %d steps (+%d warm-up), %.3f s/step, torch %s CPU"
                      % (wl["name"], kind, n, steps, warmup, dt, torch.__version__)}, dt, n


def run_reference_arm(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warm = max(1, args.steps), max(0, args.warmup)
    cb, dt, n = cpu_reference_run(wl, steps, warm, args.cpu_sample)
    line = {"impl": "reference", "metric": wl["metric"], "value": cb["value"], "unit": "samples/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warm, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "%s on the host CPU; bounded sample batch %d of the batch-%d workload"
                                   % (wl["what"], n, args.batch),
                       "bench_config": args.config, "L": wl["L"], "D": D_FEAT, "T": T_TOK, "answers": ANSWERS},
            "cpu_baseline": cb, "gpu_launches": 0,
            "e2e": {"value": cb["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    _OUT.write(json.dumps(line) + "\n")
    _OUT.flush()


# ------------------------------------------------------------------------------------------------
# GPU arm: roofline descriptions per workload
# ------------------------------------------------------------------------------------------------
def roofline_specs(wl, B, precision):
    """[(key, tag, bound, kernel, algorithmic work per launch)] -- first entry is the line's `roofline`."""
    L = wl["L"]
    s = 2 if precision == "bf16" else 4
    pool_bytes = B * L * D_FEAT * s + B * 2 * L * 4 + B * 2 * D_FEAT * 4
    pool = ("softmax_pool_fwd_regions", "hbm", "softmax_pool_fwd_kernel (softmax over the regions + 2-glimpse pooling, "
            "mhb_coAtt.py:114-121 / mfb.py:116-123)", pool_bytes)
    if wl["model"] == "mhbcoatt":
        flops = 2.0 * (B * L) * 5000 * D_FEAT * (3 if precision == "fp32" else 1)
        return [("roofline", "mfb_fused_spatial", "tensor",
                 "gemm_tcgen05_kernel<240, EPI_MFB> (img_conv1d + MFB epilogue, forward, mhb_coAtt.py:97-106)", flops),
                ("roofline_hbm_kernel",) + pool]
    if wl["model"] == "mfb":
        # degenerate softmax (mfb.py:84,118): the dense first stage is dead code and not executed; the step is the
        # region sum-pool (one read of X) plus the weight-streaming vector MFB block
        vec_bytes = 5000 * 2 * D_FEAT * s + B * 2 * D_FEAT * s + B * 5000 * (4 + 2) + B * 1000 * 4
        return [("roofline",) + pool,
                ("roofline_vector_block", "mfb_fused_vector", "hbm",
                 "gemm_tcgen05_kernel<240, EPI_MFB> (img_proj2 + MFB epilogue on pooled vectors, mfb.py:126-133): weight "
                 "streaming", vec_bytes)]
    flops = 2.0 * (B * L) * E_HIE * D_FEAT * (3 if precision == "fp32" else 1)
    aff_bytes = B * (T_TOK + L) * E_HIE * 2 + B * T_TOK * 200 * 4
    return [("roofline", "hie_img_emb", "tensor",
             "gemm_tcgen05_kernel<256, EPI_STORE> (img_emb Linear + ReLU + dropout epilogue, hieCoAtten.py:25-26)", flops),
            ("roofline_affinity", "hie_affinity", "hbm",
             "gemm_tcgen05_kernel<128, EPI_STORE> batched (C = tanh(Cq Cv^T) + dropout, hieCoAtten.py:32-33)", aff_bytes)]


def roofline_entry(spec, ktimes, ms_total, peaks):
    _, tag, bound, kernel, work = spec
    n_l, tot = ktimes.get(tag, (0, 0.0))
    if not n_l:
        return None
    avg_ms = tot / n_l
    if bound == "tensor":
        ach, peak, unit, src = work / (avg_ms * 1e-3) / 1e12, peaks["bf16_sustained"], "TFLOP/s", " (sustained cuBLAS bf16)"
    else:
        ach, peak, unit, src = work / (avg_ms * 1e-3) / 1e9, peaks["hbm"], "GB/s", " (copy bandwidth)"
    out = {"bound": bound, "kernel": kernel, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak,
           "peak_source": peaks["source"] + src, "avg_launch_ms": avg_ms, "launches": n_l,
           "share_of_step": tot / ms_total, "traffic": None,
           ("algorithmic_flops" if bound == "tensor" else "algorithmic_bytes"): work}
    if bound == "tensor":
        # the denominator is what cuBLAS sustains on this pool; a hand-written kernel may exceed it (frac > 1): the burst
        # figure bounds it from above
        out["frac_of_burst_peak"] = ach / peaks["bf16_burst"]
    return out


def attach_traffic(roof, key, B, precision):
    """DRAM bytes per launch of the same kernel from the committed `ncu --set full` capture (profiles/)."""
    if roof is None or B != 256 or precision != "bf16":
        return
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))[key]
        roof["traffic"] = tr["dram_bytes_per_launch"]
        roof["traffic_source"] = tr["source"]
        for k in ("algorithmic_bytes", "declared_extra_bytes", "declared_extra"):
            if k in tr:
                roof[k] = tr[k]
    except Exception:
        pass


# ------------------------------------------------------------------------------------------------
# GPU arm: train-step configurations (c1..c4)
# ------------------------------------------------------------------------------------------------
def run_train(args, wl):
    import torch
    import torch.distributed as dist
    from vqa_attention_networks_b200 import ops
    from vqa_attention_networks_b200.ddp import GradientAllReducer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    from vqa_attention_networks_b200.feed import bind_to_gpu_numa_node as bind_numa
    bind_numa(local)                          # before any pinned allocation: first touch on the GPU's NUMA node
    if world > 1:
        _init_process_group(dist, dev, rank, world)
    B = args.batch
    K, W = args.steps, max(3, args.warmup)
    L = wl["L"]

    model = build_model(torch, wl)
    model.precision = args.precision
    model = model.to(dev).train()
    if args.optimizer == "fused":
        from vqa_attention_networks_b200.optim import FusedAdam
        opt = FusedAdam(model.parameters(), lr=wl["lr"]).attach(model)        # solver.py:30, SURVEY 8f rank 1
    else:
        opt = torch.optim.Adam(model.parameters(), lr=wl["lr"], fused=True, capturable=bool(args.graph))   # solver.py:30
    defer = None
    if wl["model"] == "mhbcoatt" and os.environ.get("VQA_B200_DDP_DEFER", "1") == "1":
        defer = [p for n, p in model.named_parameters() if not n.startswith(("lstm.", "word_embedding."))]
    shard = bool(args.shard) and args.optimizer == "fused" and args.precision == "bf16"
    reducer = GradientAllReducer(model, defer_params=defer, shard_optimizer=opt if shard else None) if world > 1 else None
    n_sharded = sum(p.numel() for b in reducer.buckets if b.sharded for p in b.params) if reducer is not None else 0
    crit = torch.nn.KLDivLoss() if wl["target"] == "soft" else torch.nn.CrossEntropyLoss()     # solver.py:26-29

    from vqa_attention_networks_b200.train import GraphedTrainStep, TrainStep
    eager_step = TrainStep(model, crit, opt, reducer,
                           bucket_step=os.environ.get("VQA_B200_BUCKET_STEP", "1") == "1")

    # ---- device-resident inputs: two distinct batches (each batch of features >> the 126 MB L2 at batch >= 128)
    host = [synth_batch(torch, B, 1234 + 17 * rank + i, pin=True, L=L, target=wl["target"]) for i in range(2)]
    resident = [tuple(t.to(dev) for t in hb) for hb in host]
    feat_mb = host[0][0].numel() * 4 / 1e6
    l2_flush = None
    if 2 * feat_mb < 300:            # small batches (c1): two batches would fit the L2 -> flush it between steps
        l2_flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    specs = roofline_specs(wl, B, args.precision)
    roof_tags = [s_[1] for s_ in specs]
    # ---- the whole iteration captured in CUDA graphs, one per input slot (train.GraphedTrainStep): slots 0/1 hold the two
    # resident batches of `value`, all three are the H2D targets of `e2e`.  The roofline kernels stay outside the graphs
    # so that they can be bracketed with CUDA events inside the timed region.
    NSLOT = 3
    graphed, graph_error = None, os.environ.get("VQA_B200_BENCH_GRAPH_ERROR")
    slots = resident + [tuple(torch.empty_like(t) for t in resident[0]) for _ in range(NSLOT - len(resident))]
    slots[2][0].copy_(resident[0][0]); slots[2][1].copy_(resident[0][1]); slots[2][2].copy_(resident[0][2])
    if args.graph:
        try:
            if os.environ.get("VQA_B200_BENCH_FORCE_CAPTURE_FAILURE") == "1":      # exercises the fallback below
                raise RuntimeError("forced capture failure (VQA_B200_BENCH_FORCE_CAPTURE_FAILURE)")
            graphed = GraphedTrainStep(eager_step, slots, warmup=W, segment_tags=roof_tags)
        except Exception as e:
            # A failed capture leaves torch's CUDA generator and the allocator's capture pools in an undefined state:
            # keep the bench alive by starting over in a fresh interpreter without graphs (every rank takes this path,
            # the failure is deterministic), and say why in the line's config.
            graph_error = "%s: %s" % (type(e).__name__, str(e).splitlines()[0][:200])
            print("bench: CUDA-graph capture failed (%s); re-running eagerly" % graph_error, file=sys.stderr)
            _reexec_eager(graph_error)

    def train_step(i):
        """iteration on slot i (resident batch i for i < 2)"""
        if graphed is not None:
            return graphed.replay(i)
        return eager_step(*slots[i])

    for i in range(W):
        train_step(i % 2)
    barrier()

    # ---- timed region 1: `value` (inputs resident in HBM).  The roofline kernels are bracketed with CUDA events
    # live, inside this region; the full per-kernel breakdown is taken in a separate eager pass below (two event
    # records per launch cost ~1 ms of host time per step)
    ops.LaunchStats.reset(timing=True, only=roof_tags)
    if graphed is not None:
        graphed.reset_times(True)
    barrier()
    sampler.begin()
    h0 = time.perf_counter()
    if l2_flush is None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(K):
            loss = train_step(i % 2)
        e1.record()
        host_enqueue_ms = (time.perf_counter() - h0) * 1e3 / K      # host time to ENQUEUE a step (no sync inside)
        barrier()
        ms_total = e0.elapsed_time(e1)
    else:
        evs = []
        for i in range(K):
            l2_flush.fill_(i & 0xFF)                                  # 256 MB write: evicts the 126 MB L2 (untimed)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            loss = train_step(i % 2)
            b.record()
            evs.append((a, b))
        host_enqueue_ms = (time.perf_counter() - h0) * 1e3 / K
        barrier()
        ms_total = sum(a.elapsed_time(b) for a, b in evs)
    sampler.end()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"loss": loss})
    if graphed is not None:
        launches = graphed.launches * K
        ktimes = graphed.kernel_times()
        graphed.reset_times(False)
    else:
        launches = ops.LaunchStats.count
        ktimes = ops.LaunchStats.summary()
    clocks = sampler.stop() if rank == 0 else None
    # per-kernel breakdown: a few more EAGER steps with every launch bracketed (not part of `value`)
    KB = min(K, 10)
    ops.LaunchStats.reset(timing=True)
    for i in range(KB):
        (graphed._iteration(slots[i % 2]) if graphed is not None else eager_step(*slots[i % 2]))
    barrier()
    kbreak = ops.LaunchStats.summary()
    ops.LaunchStats.reset(timing=False)
    t = torch.tensor([ms_total], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_step = ms_total / K
    value = world * B * K / (ms_total / 1e3)

    # ---- timed region 2: `e2e` -- host inputs, H2D inside the timed region, the loss read back every step.
    # Headline form: the repo's own data feed (feed.ShardFeed): a packed bf16 feature shard (written here from the same
    # synthetic batches) -> pinned ring -> copy stream -> the step's static bf16 input slots, two batches ahead.
    # Conservative form (`e2e_fp32_feed`): pinned fp32 [N, L, 2048] host batches, the reference DataLoader's format.
    from vqa_attention_networks_b200 import feed as vfeed
    NS = len(slots)

    def read_losses_pipelined(run_step, steps):
        """run_step(i) -> loss tensor of step i (already ordered on the current stream).  Every loss is read back through
        pinned memory one step behind, so the host never drains the GPU queue."""
        loss_host = [torch.zeros((), dtype=torch.float32).pin_memory() for _ in range(2)]
        loss_ready = [torch.cuda.Event() for _ in range(2)]
        losses = []
        for i in range(steps):
            loss = run_step(i)
            loss_host[i % 2].copy_(loss.detach(), non_blocking=True)     # D2H read of the step's result
            loss_ready[i % 2].record()
            if i > 0:
                loss_ready[(i - 1) % 2].synchronize()
                losses.append(float(loss_host[(i - 1) % 2]))
        loss_ready[(steps - 1) % 2].synchronize()
        losses.append(float(loss_host[(steps - 1) % 2]))
        return losses

    def timed(fn):
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        out = fn()
        f1.record()
        barrier()
        t_ = torch.tensor([f0.elapsed_time(f1)], device=dev)
        if world > 1:
            dist.all_reduce(t_, op=dist.ReduceOp.MAX)
        return float(t_.item()), out

    # (a) fp32 host batches -> the fp32 static slots of `graphed` (three slots: the copy of step i+2 starts the moment the
    # copy of step i+1 ends; with two it would wait for step i to release its slot)
    copy_stream = torch.cuda.Stream(device=dev)

    def e2e_fp32(steps):
        ready = [torch.cuda.Event() for _ in range(NS)]
        step_done = [None] * NS

        def issue_copy(i):
            slot, hb = i % NS, host[i % len(host)]
            with torch.cuda.stream(copy_stream):
                if step_done[slot] is not None:
                    copy_stream.wait_event(step_done[slot])      # never overwrite inputs a queued step still reads
                for d, s_ in zip(slots[slot], hb):
                    d.copy_(s_, non_blocking=True)
                ready[slot].record(copy_stream)

        issue_copy(0)
        if steps > 1:
            issue_copy(1)

        def run(i):
            if i + 2 < steps:
                issue_copy(i + 2)
            torch.cuda.current_stream().wait_event(ready[i % NS])
            loss = train_step(i % NS)
            step_done[i % NS] = torch.cuda.Event()
            step_done[i % NS].record()
            return loss
        return read_losses_pipelined(run, steps)

    h2d_gbs = h2d_bandwidth_gbs(torch, host[0][0], dev)
    ms32, losses32 = timed(lambda: e2e_fp32(K))
    e2e_fp32_feed = {"value": world * B * K / (ms32 / 1e3), "unit": "samples/s",
                     "h2d_bytes_per_step": sum(t.numel() * t.element_size() for t in host[0]), "d2h_bytes_per_step": 4,
                     "loss": losses32[-1], "h2d_gbs_measured": h2d_gbs,
                     "note": "pinned fp32 host features + dense targets (the reference DataLoader's format), H2D on a copy "
                             "stream kept two steps ahead (3 device slots); bound by the copy itself once a step is shorter "
                             "than it"}

    # (b) the feed: shard -> pinned ring -> device
    e2e = None
    if args.precision == "bf16":
        soft = wl["target"] == "soft"
        shm, shard_path, reader = None, None, None
        for cand in ("/dev/shm", tempfile.gettempdir()):      # a small /dev/shm (container default 64 MB) must not end the run
            if not (os.path.isdir(cand) and os.access(cand, os.W_OK)):
                continue
            shard_path = os.path.join(cand, "vqa_b200_bench_%d_%d.shard" % (os.getpid(), rank))
            try:
                with vfeed.ShardWriter(shard_path, L, D_FEAT, T_TOK, ANSWERS, soft_answer=soft) as w:
                    for hb in host:
                        w.append(hb[0], hb[1], hb[2])
                reader = vfeed.ShardReader(shard_path)
                shm = cand
                break
            except OSError:
                try:
                    os.remove(shard_path)
                except OSError:
                    pass
        if reader is None:
            raise RuntimeError("bench: no writable place for the %d MB feature shard" % (2 * B * L * D_FEAT * 2 >> 20))
        slots16 = [(torch.empty((B, L, D_FEAT), dtype=torch.bfloat16, device=dev), torch.empty_like(resident[0][1]),
                    torch.empty_like(resident[0][2])) for _ in range(NS)]
        fd = vfeed.ShardFeed(reader, B, dev, device_slots=slots16, depth=2, ring_slots=4)
        for i in range(NS):                                   # real data in every slot before anything is captured
            d, _ = fd.next()
            fd.done(d)
        torch.cuda.synchronize()
        graphed16 = None
        if graphed is not None:
            try:
                graphed16 = GraphedTrainStep(eager_step, slots16, warmup=1)
            except Exception as e:
                print("bench: capture of the bf16-input step failed, e2e runs eagerly: %s" % e, file=sys.stderr)

        def run16(i):
            d, (img, q, tgt, _ql) = fd.next()
            loss = graphed16.replay(d) if graphed16 is not None else eager_step(img, q, tgt)
            fd.done(d)
            return loss

        read_losses_pipelined(run16, 3)                       # warm-up of the pipeline
        ms16, losses16 = timed(lambda: read_losses_pipelined(run16, K))
        e2e = {"value": world * B * K / (ms16 / 1e3), "unit": "samples/s", "h2d_bytes_per_step": fd.h2d_bytes_per_batch(),
               "d2h_bytes_per_step": 4, "loss": losses16[-1], "losses_read": len(losses16), "numa_node": fd.numa_node,
               "staging_gbs": fd.staging_gbs(), "ring": "pinned cache of the shard" if fd.cached else "streaming",
               "note": "feed.ShardFeed: packed bf16 [N,L,2048] feature shard (+ int32 tokens, sparse soft answers) in %s -> "
                       "pinned ring -> copy stream two batches ahead -> the step's static inputs; every step's loss is read "
                       "back through pinned memory one step behind.  bf16 mode rounds fp32 features to these very values "
                       "on the device, so results equal the fp32 feed's" % shm}
        fd.close()
        del graphed16, fd, reader
        try:
            os.remove(shard_path)
        except OSError:
            pass
    if e2e is None:                                           # fp32 mode computes with fp32 features: the fp32 feed it is
        e2e = dict(e2e_fp32_feed)

    # ---- extra (not the headline): the hot-path block alone (SURVEY 8d "block-only"): fused_block forward + backward
    # with the question states precomputed, i.e. everything the north_star path owns and nothing else
    block = None
    if hasattr(model, "fused_block"):
        qf = [model.question_features(r[1]).detach().requires_grad_(True) for r in resident]
        cotb = torch.randn(B, 2000 if wl["model"] == "mhbcoatt" else 1000, device=dev)

        def block_step(i):
            for p_ in model.parameters():
                p_.grad = None
            if reducer is not None:
                reducer.prepare()                    # gradient destinations inside the buckets are handed out once per step
            out = model.fused_block(resident[i % 2][0], qf[i % 2])
            out.backward(cotb)

        for i in range(3):
            block_step(i)
        barrier()
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        b0.record()
        for i in range(K):
            block_step(i)
        b1.record()
        barrier()
        block_ms = b0.elapsed_time(b1) / K
        block = {"ms_per_step": block_ms, "samples_per_s_per_gpu": B / (block_ms / 1e3),
                 "note": "fused_block forward+backward only (question attention, MFB blocks, co-attention, train-mode "
                         "dropout); LSTM / embedding / classifier / Adam excluded"}
        if wl["model"] == "mhbcoatt" and L == 196:
            # SURVEY 8a: algorithmic dense FLOPs of the block, forward + backward, each GEMM once: 9.180 GFLOP per sample
            tf = 9.180e9 * B / (block_ms * 1e-3) / 1e12
            block["algorithmic_tflops"] = tf
            block["tensor_roofline_frac"] = tf / measured_peaks()["bf16_sustained"]

    # ---- exposed (non-overlapped) time of the gradient exchange: the same captured iteration once more WITHOUT its
    # collectives (reducer.dry_run: same bucket writes, shard updates and weight copies, no NCCL call), timed the same way;
    # exposed = ms_per_step - that.  Runs last (after `e2e`): not part of any reported rate, and the ranks' weights drift
    # apart from here on.
    comm = None
    if world > 1 and reducer is not None and graphed is not None and os.environ.get("VQA_B200_BENCH_DRY", "1") == "1":
        saved = [(m, m.seed_counter) for m in model.modules() if hasattr(m, "seed_counter")]
        g2 = None
        try:
            reducer.dry_run = True
            g2 = GraphedTrainStep(eager_step, slots, warmup=2)
            for i in range(3):
                g2.replay(i % 2)
            barrier()
            d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            d0.record()
            for i in range(K):
                g2.replay(i % 2)
            d1.record()
            barrier()
            td = torch.tensor([d0.elapsed_time(d1) / K], device=dev)
            dist.all_reduce(td, op=dist.ReduceOp.MAX)
            ms_dry = float(td.item())
            comm = {"ms_per_step_without_collectives": ms_dry, "exposed_comm_ms": ms_step - ms_dry,
                    "how": "same captured iteration with the reducer's collectives elided (dry_run), max over ranks"}
        except Exception as e:                                   # the headline numbers do not depend on this leg
            comm = {"error": "%s: %s" % (type(e).__name__, str(e).splitlines()[0][:160])}
        finally:
            reducer.dry_run = False
            for m, c in saved:
                m.seed_counter = c
            del g2
            gc.collect()

    graph_desc = (("whole iteration captured (train.GraphedTrainStep), %d graph segments per step; roofline kernels "
                   "launched between segments" % len(graphed.programs[0])) if graphed is not None
                  else ("off" + ("; capture failed: " + graph_error if graph_error else "")))
    graphed = None                         # drop the captured graphs (they hold NCCL kernels) before any teardown
    if rank != 0:
        _shutdown(torch, dist, world)
        return

    peaks = measured_peaks()
    roofs = {}
    for spec in specs:
        roofs[spec[0]] = roofline_entry(spec, ktimes, ms_total, peaks)
    if wl["model"] == "mhbcoatt":
        attach_traffic(roofs.get("roofline"), "mfb_fused_spatial", B, args.precision)
        attach_traffic(roofs.get("roofline_hbm_kernel"), "softmax_pool_fwd_regions", B, args.precision)
    breakdown = {k: {"launches": v[0], "ms_per_step": v[1] / KB} for k, v in sorted(kbreak.items(), key=lambda kv: -kv[1][1])}

    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        cpu_baseline, _, _ = cpu_reference_run(wl, 2, 1, args.cpu_sample, budget_s=60.0)

    allreduce_bytes = reducer.bytes_per_step() if reducer is not None else 0
    line = {"metric": wl["metric"], "value": value, "unit": "samples/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if args.precision == "bf16" else "f32(bf16x3)", "data": "synthetic",
            "config": {"workload": "%s, batch %d per GPU, %dx2048 features, 26 tokens, 15k vocab, 3000 answers"
                                   % (wl["what"], B, L),
                       "bench_config": args.config, "global_batch": B * world, "parallelism": "dp%d" % world,
                       "l2_policy": ("two alternating batches; %.0f MB of features per batch > 126 MB L2" % feat_mb)
                       if l2_flush is None else "256 MB buffer written between timed steps (L2 flush); each step timed "
                                                "with its own CUDA events",
                       "precision": args.precision,
                       "optimizer": "FusedAdam (vqa_b200_adam_step)" if args.optimizer == "fused" else "torch.optim.Adam(fused=True)",
                       "cuda_graph": graph_desc,
                       "allreduce_bytes_per_step": allreduce_bytes,
                       "gradient_exchange": (("reduce-scatter + Adam on the shard + all-gather of the bf16 weight copies for "
                                              "%d of %d parameters, all-reduce for the rest; %d wire bytes per rank and step"
                                              % (n_sharded, sum(p.numel() for p in model.parameters()),
                                                 reducer.wire_bytes_per_step())) if n_sharded else
                                             ("bucketed all-reduce, %d wire bytes per rank and step"
                                              % reducer.wire_bytes_per_step())) if reducer is not None else "none (1 GPU)"},
            "e2e": e2e, "e2e_fp32_feed": e2e_fp32_feed, "hot_path_block": block,
            "gpu_launches": launches, "host_enqueue_ms_per_step": host_enqueue_ms, "clocks": clocks}
    if comm is not None:
        line["gradient_exchange_exposed"] = comm
    line.update(roofs)
    line["cpu_baseline"] = cpu_baseline
    line["kernel_breakdown_ms_per_step"] = breakdown
    line["kernel_breakdown_note"] = ("eager steps outside the timed region, every launch bracketed by CUDA events: exact for "
                                     "the GPU-bound kernels; entries of many short launches (recurrence steps, casts) "
                                     "include the host's launch gaps and overstate their share of the captured step")
    _OUT.write(json.dumps(line) + "\n")
    _OUT.flush()
    _shutdown(torch, dist, world)


# ------------------------------------------------------------------------------------------------
# GPU arm: inference sweep (c5)
# ------------------------------------------------------------------------------------------------
def run_infer(args, wl):
    """MHBCoAtt eval forward, L = 100, global batch b in {1, 2, 4, ..., --batch}: rank r takes rows
    [r b / P, (r+1) b / P) (ranks without rows idle for that b); no communication on the data path.  One CUDA-graph
    replay per step (inference.GraphedForward).  `value` is the throughput at the largest batch."""
    import torch
    import torch.distributed as dist
    from vqa_attention_networks_b200 import ops
    from vqa_attention_networks_b200.inference import GraphedForward

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    from vqa_attention_networks_b200.feed import bind_to_gpu_numa_node as bind_numa
    numa_node = bind_numa(local)
    if world > 1:
        _init_process_group(dist, dev, rank, world)
    K, W = args.steps, max(3, args.warmup)
    L = wl["L"]
    model = build_model(torch, wl)
    model.precision = args.precision
    model = model.to(dev).eval()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sizes = []
    b = 1
    while b <= args.batch:
        sizes.append(b)
        b *= 2
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    sweep, roof, e2e_last, launches_total = [], None, None, 0
    peaks = measured_peaks()
    for gb in sizes:
        lo, hi = rank * gb // world, (rank + 1) * gb // world
        n = hi - lo
        ms_dev = ms_e2e = 0.0
        launches = 0
        if n > 0:
            host = [synth_batch(torch, n, 4321 + 31 * rank + i, pin=True, L=L, target="hard")[:2] for i in range(2)]
            res = [tuple(t.to(dev) for t in hb) for hb in host]
            ops.LaunchStats.reset(timing=False)
            with torch.no_grad():
                model(*res[0])                                    # eager pass: counts the launches one forward makes
            launches = ops.LaunchStats.count
            g = GraphedForward(model, res[0][0], res[0][1], warmup=W)
            for i in range(W):
                g(*res[i % 2])
        barrier()
        if rank == 0 and gb == sizes[-1]:
            sampler.begin()
        if n > 0:
            # `value`: inputs resident; the L2 is flushed between replays (a batch of features fits the 126 MB L2 up to
            # batch ~300), every replay timed with its own events
            evs = []
            for i in range(K):
                flush.fill_(i & 0xFF)
                a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                g.img.copy_(res[i % 2][0], non_blocking=True)
                g.q.copy_(res[i % 2][1], non_blocking=True)
                a.record()
                g.graph.replay()
                b_.record()
                evs.append((a, b_))
            torch.cuda.synchronize()
            ms_dev = sum(a.elapsed_time(b_) for a, b_ in evs) / K
        if rank == 0 and gb == sizes[-1]:
            sampler.end()
            if args.dump_outputs:
                dump_outputs(args.dump_outputs, {"out": g.out})
        if n > 0:
            # `e2e`: pinned host inputs -> H2D -> replay -> argmax -> D2H of the predicted answers, every step
            pred_host = torch.zeros(n, dtype=torch.int64).pin_memory()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            f0.record()
            for i in range(K):
                out = g(host[i % 2][0], host[i % 2][1])
                pred_host.copy_(out.argmax(1), non_blocking=True)
            f1.record()
            torch.cuda.synchronize()
            ms_e2e = f0.elapsed_time(f1) / K
            # roofline of the fused img_conv1d + MFB kernel at the largest batch: one more eager, bracketed pass
            if gb == sizes[-1]:
                ops.LaunchStats.reset(timing=True, only=["mfb_fused_spatial"])
                with torch.no_grad():
                    for i in range(3):
                        flush.fill_(i)
                        model(*res[i % 2])
                torch.cuda.synchronize()
                kt = ops.LaunchStats.summary()
                ops.LaunchStats.reset(timing=False)
                flops = 2.0 * (n * L) * 5000 * D_FEAT * (3 if args.precision == "fp32" else 1)
                roof = roofline_entry(("roofline", "mfb_fused_spatial", "tensor",
                                       "gemm_tcgen05_kernel<240, EPI_MFB> (img_conv1d + MFB epilogue, inference: no keep "
                                       "tensor, no dropout)", flops), kt, ms_dev * 3, peaks)
            del g, res, host
        t = torch.tensor([ms_dev, ms_e2e], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_dev, ms_e2e = float(t[0]), float(t[1])
        if n > 0 and rank == 0:
            launches_total = launches
        sweep.append({"global_batch": gb, "ms": ms_dev, "samples_per_s": gb / (ms_dev / 1e3) if ms_dev > 0 else 0.0,
                      "e2e_ms": ms_e2e, "e2e_samples_per_s": gb / (ms_e2e / 1e3) if ms_e2e > 0 else 0.0})
        if gb == sizes[-1]:
            per_rank = max(1, gb // world)
            e2e_last = {"value": gb / (ms_e2e / 1e3), "unit": "samples/s",
                        "h2d_bytes_per_step": per_rank * (L * D_FEAT * 4 + T_TOK * 8), "d2h_bytes_per_step": per_rank * 8,
                        "note": "per rank and step: pinned fp32 host features + token ids H2D, graph replay, argmax, "
                                "predicted answer ids D2H; no overlap between copy and compute (latency path)",
                        "numa_node": numa_node}
    clocks = sampler.stop() if rank == 0 else None
    if rank != 0:
        _shutdown(torch, dist, world)
        return
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        cpu_baseline, _, _ = cpu_reference_run(wl, 2, 1, args.cpu_sample, budget_s=60.0)
    last = sweep[-1]
    line = {"metric": wl["metric"], "value": last["samples_per_s"], "unit": "samples/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": last["ms"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "bf16" if args.precision == "bf16" else "f32(bf16x3)", "data": "synthetic",
            "config": {"workload": "%s over %d GPU(s), 100x2048 features, 26 tokens, 15k vocab, 3000 answers; value at "
                                   "global batch %d" % (wl["what"], world, last["global_batch"]),
                       "bench_config": args.config, "global_batch": last["global_batch"], "parallelism": "dp%d" % world,
                       "l2_policy": "256 MB buffer written between timed replays (L2 flush); each replay timed with its "
                                    "own CUDA events", "precision": args.precision},
            "e2e": e2e_last, "gpu_launches": launches_total * K, "launches_per_forward": launches_total,
            "clocks": clocks, "roofline": roof, "cpu_baseline": cpu_baseline, "sweep": sweep}
    _OUT.write(json.dumps(line) + "\n")
    _OUT.flush()
    _shutdown(torch, dist, world)


def _shutdown(torch, dist, world):
    """End of a rank.  CUDA graphs that contain NCCL kernels must be gone before the communicator is destroyed
    (ncclCommDestroy blocks for ever on a communicator that live graphs still reference: measured, N = 2), and a teardown
    must never cost the run its result: the JSON line is already out, so a watchdog ends the process if NCCL does not
    come back."""
    import gc
    import threading
    _OUT.flush()
    if world <= 1:
        return
    threading.Timer(20.0, lambda: os._exit(0)).start()
    gc.collect()
    torch.cuda.synchronize()
    try:
        dist.barrier()
        dist.destroy_process_group()
    finally:
        os._exit(0)


_REAL_STDOUT_FD = None


def _init_process_group(dist, dev, rank, world):
    """NCCL process group from the launcher's environment.  In the interpreter that _reexec_eager() started, the
    rendezvous store of the torchrun agent still holds the keys of the first attempt (the NCCL unique id among them):
    the retry registers under its own prefix instead of reading those."""
    if world == 2:
        # Two ranks exchange over plain P2P rings, whose bandwidth scales with the number of channels: measured exposed
        # time of the exchange 0.635 ms (NCCL's default) -> 0.590 (>= 32 CTAs) -> 0.545 (>= 64) per step, caps below the
        # default are worse (tools/nccl_sweep.sh; DESIGN.md 6).  Larger worlds keep NCCL's choice (N = 4: no gain, 0.75 ->
        # 0.78 ms).  An explicit NCCL_MIN_CTAS in the environment wins.
        os.environ.setdefault("NCCL_MIN_CTAS", "64")
    if os.environ.get("VQA_B200_BENCH_GRAPH_ERROR") and os.environ.get("TORCHELASTIC_USE_AGENT_STORE") == "True":
        store = dist.TCPStore(os.environ["MASTER_ADDR"], int(os.environ["MASTER_PORT"]), world, is_master=False)
        dist.init_process_group("nccl", store=dist.PrefixStore("vqa_b200_eager_retry", store), rank=rank,
                                world_size=world, device_id=dev)
    else:
        dist.init_process_group("nccl", device_id=dev)


def _protect_stdout():
    """Libraries (NCCL's version banner, warnings) must not share stdout with the ONE JSON line: route fd 1 to stderr
    for the whole run and return a writer on the real stdout."""
    global _REAL_STDOUT_FD
    real = os.dup(1)
    os.dup2(2, 1)
    _REAL_STDOUT_FD = real
    return os.fdopen(real, "w")


def _reexec_eager(reason):
    """Replace this process by `bench.py ... --graph 0` (same rank environment, the real stdout back on fd 1)."""
    sys.stderr.flush()
    if _REAL_STDOUT_FD is not None:
        os.dup2(_REAL_STDOUT_FD, 1)
    os.environ["VQA_B200_BENCH_GRAPH_ERROR"] = reason
    os.environ.pop("VQA_B200_BENCH_FORCE_CAPTURE_FAILURE", None)
    argv = [a for a in sys.argv]
    os.execv(sys.executable, [sys.executable] + argv + ["--graph", "0"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (c5: largest global batch); 0 = the config's own")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--cpu-sample", type=int, default=64, help="batch of the bounded CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--shard", type=int, default=1, help="N > 1: 1 = sharded optimizer (reduce-scatter / Adam on the shard / "
                                                         "all-gather of bf16 weights), 0 = all-reduce + full update")
    ap.add_argument("--graph", type=int, default=1, help="1: capture the train iteration in CUDA graphs (default); 0: eager")
    ap.add_argument("--optimizer", default="fused", choices=["fused", "torch"],
                    help="fused: this repo's multi-tensor Adam (also refreshes the bf16 weight copies); torch: stock")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    wl = WORKLOADS[args.config]
    if args.batch <= 0:
        args.batch = wl["batch"]
    global _OUT
    _OUT = _protect_stdout()
    if args.impl == "reference":
        run_reference_arm(args, wl)
    elif wl["target"] is None:
        run_infer(args, wl)
    else:
        run_train(args, wl)


if __name__ == "__main__":
    main()
