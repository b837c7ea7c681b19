#!/usr/bin/env python
"""Benchmark of the gradient-inversion hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--config C] [--dump-outputs DIR]   # product arm: the sm_100a engine
    python bench.py --impl reference --steps K --warmup W [--config C]     # reference arm: CPU restatement of the reference loop

A "step" is one iteration of ``OptimizationBasedAttacker._run_trial`` (closure + optimiser step + projection + best-so-far)
on one candidate batch.  ``--config`` picks the BASELINE.json configuration (default 2, the one the metric is quoted on):

    1  invertinggradients, ConvNet(64) / CIFAR-10 shape, 1 image
    2  invertinggradients, torchvision ResNet-18 (397 classes), 1 x 3x224x224
    3  see-through-gradients, ResNet-50, 8 x 3x224x224 (user buffers, DeepInversion prior)
    4  modern (cosine, TV double opponents) on a ResNet-18 FedAvg update: 4 points, 4 local steps
    5  TAG (joint data + label optimisation), 3-layer transformer (50257 tokens, 96 dims), 32 positions

With N GPUs every rank runs an independent restart (trial) of the same workload, no data-path collective (weak scaling);
value = N*K / max-over-ranks device time.  The ``e2e`` leg goes through ``prepare_attack(...).reconstruct(...)`` with
``restarts.num_trials = N`` (trial k on rank k, NCCL MIN select + broadcast of the winner) from pinned host buffers.
Prints ONE JSON line on rank 0.
"""
import argparse
import copy
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    1: dict(name="BASELINE config 1: invertinggradients, ConvNet(width 64, 10 classes, random init), synthetic 3x32x32 batch=1",
            metric="reconstruction iters/sec (ConvNet-64 32x32, invertinggradients)", attack="invertinggradients", e2e_steps=24000, ref_steps=40),
    2: dict(name="BASELINE config 2: invertinggradients, torchvision ResNet-18 (397 classes, random init), synthetic 3x224x224 batch=1",
            metric="reconstruction iters/sec (ResNet-18 224x224, invertinggradients)", attack="invertinggradients", e2e_steps=24000, ref_steps=20),
    3: dict(name="BASELINE config 3: see-through-gradients (euclidean, TV, norm, DeepInversion on 53 BN layers, yin labels), torchvision "
                 "ResNet-50 (397 classes, random init, user buffers), synthetic 3x224x224 batch=8",
            metric="reconstruction iters/sec (ResNet-50 224x224 batch 8, see-through-gradients)", attack="seethroughgradients", e2e_steps=800,
            ref_steps=3),
    4: dict(name="BASELINE config 4: modern (cosine, soft sign, TV double opponents; features prior off -- the reference crashes with it under "
                 "FedAvg) on a torchvision ResNet-18 FedAvg update (4 points, 4 local steps x 1, lr 1e-3), synthetic 3x224x224",
            metric="reconstruction iters/sec (ResNet-18 224x224 FedAvg 4 steps, modern)", attack="modern", e2e_steps=1200, ref_steps=4),
    5: dict(name="BASELINE config 5: TAG (tag-euclidean, AdamW, clip 1.0, joint label optimisation), TransformerModel(50257 tokens, 96 dims, "
                 "8 heads, 1536 hidden, 3 layers), synthetic tokens seq=32 batch=1",
            metric="reconstruction iters/sec (transformer3 seq 32, TAG)", attack="tag", e2e_steps=1000, ref_steps=10),
}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            d = json.load(fh)
        return dict(hbm_gbs=d.get("hbm_gbs", 6650.0), bf16_tflops=d.get("bf16_tflops", 1590.0),
                    bf16_tflops_sustained=d.get("bf16_tflops_sustained", 1400.0), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


class ClockSampler:
    """SM clock and throttle reasons sampled through NVML every ~2 ms while the timed region runs (nvidia-smi's 100 ms loop
    misses a 30 ms region); falls back to one nvidia-smi query when NVML is unavailable."""

    def __init__(self, index):
        self.index, self.rows, self.stop, self.thread = index, [], threading.Event(), None
        self.max_mhz = None

    def __enter__(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.nv = None
        return self

    def _loop(self):
        nv = self.nv
        while not self.stop.is_set():
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM))
                reasons = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle)) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                self.rows.append((sm, reasons))
            except Exception:  # noqa: BLE001
                break
            time.sleep(0.002)

    def __exit__(self, *exc):
        self.stop.set()
        if self.thread is not None:
            self.thread.join(timeout=1)

    def summary(self):
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        sm = sorted(r[0] for r in self.rows)
        reasons = set()
        for _, bits in self.rows:
            for bit, name in names.items():
                if bits & bit:
                    reasons.add(name)
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=self.max_mhz, reasons=sorted(reasons), samples=len(sm),
                    source="nvml, 2 ms period, during the timed region")


# ---- workloads -----------------------------------------------------------------------------------------------------------
def build_case(config, seed=233):
    """(model, loss_fn, server_payload, shared_data, true_user_data, cfg_attack) for one BASELINE configuration (SURVEY 8d)."""
    import torch

    from breaching_b200 import get_attack_config, synthetic

    torch.manual_seed(seed + 1)  # breaching/utils.py:159-167 seeding recipe (CPU generator part)
    w = WORKLOADS[config]
    over = {}
    if config == 1:
        case = synthetic.make_case("convnet", "cifar", batch=1, seed=seed)
    elif config == 2:
        case = synthetic.make_case("resnet18", "imagenet", batch=1, seed=seed)
    elif config == 3:
        case = synthetic.make_case("resnet50", "imagenet", batch=8, seed=seed, user_buffers=True)
    elif config == 4:
        case = synthetic.make_fedavg_case("resnet18", "imagenet", num_data_points=4, steps=4, data_per_step=1, lr=1e-3, seed=seed)
        over = {"regularization.features.scale": 0.0}
    elif config == 5:
        case = synthetic.make_text_case(batch=1, seq_len=32, seed=seed, ntokens=50257, ninp=96, nhead=8, nhid=1536, nlayers=3)
    else:
        raise SystemExit(f"unknown --config {config}")
    return (*case, get_attack_config(w["attack"], over))


def candidate_shape(config, payload, shared):
    meta = payload[0]["metadata"]
    n = shared[0]["metadata"]["num_data_points"]
    return (n, *meta.shape)


def gemm_ops(prog, backend="simt"):
    """Conv / linear layers of the program as GEMM geometries.  On the tensor-core back end the candidate-fed convolution runs as
    a 1x1 convolution over the unfolded candidate (csrc/stem_cols.cu: K = R*S*Ci padded to a multiple of 64); its *algorithmic*
    MACs stay those of the original layer."""
    from breaching_b200 import compiler as C

    out = []
    for op in prog.ops:
        if op.kind not in (C.OP_CONV, C.OP_LINEAR):
            continue
        ti, to = prog.tensors[op.tin], prog.tensors[op.tout]
        if op.kind == C.OP_LINEAR:
            g = (ti.N, 1, 1, ti.C * ti.H * ti.W, to.C, 1, 1, 0)
        else:
            g = (ti.N, ti.H, ti.W, ti.C, to.C, op.R, op.stride, op.pad)
        Ho, Wo = (to.H, to.W) if op.kind == C.OP_CONV else (1, 1)
        macs = g[0] * Ho * Wo * g[4] * g[5] * g[5] * g[3]
        if backend == "tc" and op.kind == C.OP_CONV and op.tin == 0 and ti.C <= 4 and to.C % 64 == 0 and os.environ.get("BRE_STEM_COLS", "1") != "0":
            g = (ti.N, Ho, Wo, ((op.R * op.R * ti.C + 63) // 64) * 64, to.C, 1, 1, 0)
        out.append(dict(first=op.tin == 0, geom=g, Ho=Ho, Wo=Wo, macs=macs))
    return out


def algorithmic_flops(prog, local_steps=0):
    """Conv / linear FLOPs of one iteration (SURVEY 8d, 7.3): per layer fprop + wgrad + dgrad + dual tangent fprop + dual tangent
    dgrad = 7 contractions; the layer fed by the candidate needs no first-backward dgrad and no `W . a_dot` term = 5.  FedAvg
    with K local steps: K times that, plus the dual-source tangent wgrad (2, first layer 1) of steps 2..K."""
    ops = gemm_ops(prog)
    F = sum(o["macs"] for o in ops)
    F1 = sum(o["macs"] for o in ops if o["first"])
    per_step = 2.0 * (7 * F - 2 * F1)
    if local_steps > 0:
        return local_steps * per_step + (local_steps - 1) * 2.0 * (2 * F - F1)
    return per_step


def gemm_family_roofline(dev, prog, backend, local_steps=0):
    """Live device time of the dominant kernel family -- the conv/linear implicit GEMMs -- for exactly the launches one
    iteration issues (per layer: fprop, wgrad, dgrad, dual-source tangent fprop, dual-source tangent dgrad; FedAvg: per local
    step, plus the dual-source tangent wgrad), replayed from one CUDA graph through the C ABI (`bre_conv_gemm`, the engine's
    own dispatch rule) and timed with CUDA events on the launching stream.  Operands of one replay exceed the 126 MB L2 for the
    224x224 configurations, so a replay does not run L2-hot."""
    import torch

    from breaching_b200 import engine as E

    be = 2 if backend == "tc" else 0
    launches, flops, keep = [], 0.0, []
    for o in gemm_ops(prog, backend):
        N, H, W, Ci, Co, R, st, pd = o["geom"]
        Ho, Wo = o["Ho"], o["Wo"]
        x, x2 = (torch.randn(N, H, W, Ci, device=dev) for _ in range(2))
        w, w2 = (torch.randn(Co, R, R, Ci, device=dev) for _ in range(2))
        dy, dy2 = (torch.randn(N, Ho, Wo, Co, device=dev) for _ in range(2))
        out_f, out_d, out_w = torch.empty(N, Ho, Wo, Co, device=dev), torch.empty(N, H, W, Ci, device=dev), torch.empty(Co, R, R, Ci, device=dev)
        keep += [x, x2, w, w2, dy, dy2, out_f, out_d, out_w]
        g = (N, H, W, Ci, Co, R, R, st, pd)
        f1 = 2.0 * o["macs"]
        first = o["first"]
        per_step = []
        per_step.append((lambda x=x, w=w, o_=out_f, g=g: E.conv_gemm(0, x, w, o_, *g, backend=be), f1))
        per_step.append((lambda x=x, dy=dy, o_=out_w, g=g: E.conv_gemm(2, x, dy, o_, *g, backend=be), f1))
        if not first:
            per_step.append((lambda dy=dy, w=w, o_=out_d, g=g: E.conv_gemm(1, dy, w, o_, *g, backend=be), f1))
            per_step.append((lambda x=x, w=w, x2=x2, w2=w2, o_=out_f, g=g: E.conv_gemm(0, x, w, o_, *g, a2=x2, w2=w2, backend=be), 2 * f1))
        else:
            per_step.append((lambda x=x, w=w, o_=out_f, g=g: E.conv_gemm(0, x, w, o_, *g, backend=be), f1))
        per_step.append((lambda dy=dy, w=w, dy2=dy2, w2=w2, o_=out_d, g=g: E.conv_gemm(1, dy, w, o_, *g, a2=dy2, w2=w2, backend=be), 2 * f1))
        reps = max(local_steps, 1)
        for _ in range(reps):
            launches += per_step
        if local_steps > 1:
            tw = (lambda x=x, dy=dy, x2=x2, dy2=dy2, o_=out_w, g=g: E.conv_gemm(2, x, dy, o_, *g, a2=None if first else x2, w2=None if first else dy2,
                                                                              backend=be), f1 if first else 2 * f1)
            launches += [tw] * (local_steps - 1)
    flops = sum(f for _, f in launches)
    for fn, _ in launches:
        fn()
    torch.cuda.synchronize(dev)
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            for fn, _ in launches:
                fn()
    torch.cuda.synchronize(dev)
    graph.replay()
    torch.cuda.synchronize(dev)
    reps = 5
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        graph.replay()
    e1.record()
    e1.synchronize()
    ms = e0.elapsed_time(e1) / reps
    del keep
    return dict(n_launches=len(launches), flops=flops, ms_total=ms, ms_per_launch=ms / len(launches), tflops=flops / (ms * 1e-3) / 1e12)


def matching_reduction_roofline(dev, n_params):
    """Isolated device time of the matching-reduction kernel (the HBM-bound kernel the north star names): the bare kernel is
    captured 16x into a CUDA graph over rotating (G, g) buffer pairs whose total exceeds the 126 MB L2, so every launch streams
    from HBM; the replay is timed with CUDA events on the launching stream."""
    import torch

    from breaching_b200 import engine as E

    peaks = measured_peaks()
    npairs = max(4, int(2 * 126e6 / (8 * n_params)) + 1)
    pairs = [(torch.randn(n_params, device=dev), torch.randn(n_params, device=dev)) for _ in range(npairs)]
    E.match_reduce(*pairs[0])
    reps = max(16, npairs)
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            for i in range(reps):
                E.match_reduce(*pairs[i % npairs], readback=False)
    torch.cuda.synchronize(dev)
    graph.replay()
    torch.cuda.synchronize(dev)
    replays = 5
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(replays):
        graph.replay()
    e1.record()
    e1.synchronize()
    ms = e0.elapsed_time(e1) / (reps * replays)
    out = dict(bound="hbm", achieved=8.0 * n_params / (ms * 1e-3) / 1e9, peak=peaks["hbm_gbs"], unit="GB/s", kernel="match_reduce_kernel",
               ms=ms, peak_source=peaks["source"], algorithmic_bytes=8 * n_params,
               traffic=(91086080 + 2710784) if n_params == 11_380_173 else None,
               note=f"mean of {replays} graph replays of {reps} launches over {npairs} rotating buffer pairs (cold in L2); includes "
                    "inter-kernel gaps; traffic = dram read+write bytes of one ncu --set full capture (profiles/r2_match_reduce_summary.txt)")
    out["frac"] = out["achieved"] / out["peak"]
    return out


# ---- the reference algorithm (oracle port) ------------------------------------------------------------------------------------
def make_oracle(config, case, device):
    """The reference loop for this configuration as restated in oracle/restate.py (same torch ops as the reference), on `device`."""
    import torch

    from oracle import restate

    model, loss_fn, payload, shared, true, cfg = case
    meta = payload[0]["metadata"]
    dev = torch.device(device)
    m = copy.deepcopy(model)
    if shared[0]["buffers"] is not None:                      # base_attack.py:178-181: user buffers, eval mode
        for buf, src in zip(m.buffers(), shared[0]["buffers"]):
            buf.data.copy_(src)
    m = m.to(dev).eval()
    grads = [g.to(dev) for g in shared[0]["gradients"]]
    if config == 5:                                           # base_attack.py:76-128: optimise in embedding space
        names = [n for n, _ in m.named_parameters()]
        grads.pop(names.index("encoder.weight"))
        m.encoder = torch.nn.Identity()
        orc = restate.JointTrialOracle(m, loss_fn, cfg, grads, None, torch.tensor(0.0, device=dev), torch.tensor(1.0, device=dev))
        gen = torch.Generator().manual_seed(0)
        x0 = (torch.randn(1, 32, 96, generator=gen) * 0.1).clamp(-0.1, 0.1).to(dev)
        l0 = (torch.randn(1, 32, meta.vocab_size, generator=gen) * 0.1).clamp(-0.1, 0.1).to(dev)
        return orc, (lambda n: orc.run_joint(x0, l0, iterations=n))
    dm = torch.tensor(meta.mean, device=dev)[None, :, None, None]
    ds = torch.tensor(meta.std, device=dev)[None, :, None, None]
    n = shared[0]["metadata"]["num_data_points"]
    local = shared[0]["metadata"]["local_hyperparams"]
    if local is not None:
        local = dict(local, labels=[l.to(dev) for l in local["labels"]])
        labels = torch.cat(local["labels"])
    else:
        labels = restate.recover_labels(cfg.label_strategy, shared, n).to(dev)
    orc = restate.TrialOracle(m, loss_fn, cfg, grads, labels, dm, ds, local_hyperparams=local)
    x0 = torch.randn(candidate_shape(config, payload, shared), generator=torch.Generator().manual_seed(0)).to(dev)
    return orc, (lambda k: orc.run(x0, iterations=k))


def oracle_iters_per_sec(config, case, device, warmup, steps):
    import torch

    orc, run = make_oracle(config, case, device)
    dev = torch.device(device)
    if dev.type == "cuda":
        old = torch.backends.cudnn.benchmark
        torch.backends.cudnn.benchmark = True                 # case/impl/default.yaml:12
    try:
        if warmup > 0:
            run(warmup)
        if dev.type == "cuda":
            torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        run(steps)
        if dev.type == "cuda":
            torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
    finally:
        if dev.type == "cuda":
            torch.backends.cudnn.benchmark = old
        orc.close()
    return steps / dt, dt


def cpu_thread_sweep(config, case, budget_s=12.0):
    """The reference's CPU path with the thread count that suits this host best: 64 threads on a 128-way SMT box were *slower*
    than 8-16 in round 1 (oversubscription).  Tries 8/16/32/64 (bounded by the core count), one warm-up + a few iterations each
    inside a time budget; returns (best_threads, {threads: it/s})."""
    import torch

    ncpu = os.cpu_count() or 8
    candidates = sorted({t for t in (8, 16, 32, 64) if t <= ncpu} | {min(ncpu, 8)})
    default = torch.get_num_threads()
    results = {}
    t_start = time.perf_counter()
    for t in candidates:
        torch.set_num_threads(t)
        try:
            its, dt = oracle_iters_per_sec(config, case, "cpu", 1, 2 if config in (3, 4) else 3)
        except Exception as exc:  # noqa: BLE001
            results[t] = f"failed: {exc}"
            continue
        results[t] = its
        if time.perf_counter() - t_start > budget_s and len([v for v in results.values() if isinstance(v, float)]) >= 2:
            break
    ok = {t: v for t, v in results.items() if isinstance(v, float)}
    best = max(ok, key=ok.get) if ok else default
    torch.set_num_threads(best)
    return best, results


# ---- product arm ------------------------------------------------------------------------------------------------------------
class EngineRunner:
    """Device-resident trial of configurations 1-5 behind `warm(n)` / `timed(n) -> ms`."""

    def __init__(self, config, case, dev, backend, rank):
        import torch

        from breaching_b200.engine import Engine
        from breaching_b200.schedule import lr_table

        model, loss_fn, payload, shared, true, cfg = case
        meta = payload[0]["metadata"]
        self.cfg, self.config = cfg, config
        opt = cfg.optim
        table = lr_table(opt.step_size, opt.step_size_decay, opt.warmup, opt.max_iterations)
        self.history_cap = len(table)  # the engine keeps the objective of the first len(table) iterations
        torch.manual_seed(1000 + rank)  # every rank = an independent restart
        local = shared[0]["metadata"]["local_hyperparams"]
        self.local_steps = 0 if local is None else int(local["steps"])
        if config == 5:
            from breaching_b200 import compiler
            from breaching_b200.attacks import host

            m = copy.deepcopy(model).to(dev).eval()
            sh = [dict(shared[0], gradients=[g.to(dev) for g in shared[0]["gradients"]])]
            host.prepare_for_text_data([m], sh, "run-embedding")
            prog = compiler.compile_transformer(m, 1, 32)
            self.eng = Engine(None, (32, 96, 1, 1), cfg, dev, backend=backend, program=prog)
            self.eng.load_model(params=[p.detach() for p in m.parameters()])
            L = len(sh[0]["gradients"])
            self.eng.load_targets(sh[0]["gradients"], torch.zeros(32, dtype=torch.long), tensor_weights=torch.arange(L, 0, -1, dtype=torch.float32) / L)
            x0 = (torch.randn(32, 96, 1, 1, device=dev) * 0.1).clamp(-0.1, 0.1)
            l0 = (torch.randn(1, 32, meta.vocab_size, device=dev) * 0.1).clamp(-0.1, 0.1)
            self.eng.begin_joint_trial(x0, l0, table)
            self.n_params = sum(g.numel() for g in sh[0]["gradients"])
        else:
            m = copy.deepcopy(model)
            if shared[0]["buffers"] is not None:
                for buf, src in zip(m.buffers(), shared[0]["buffers"]):
                    buf.data.copy_(src)
            m = m.to(dev).eval()
            shape = candidate_shape(config, payload, shared)
            prog_shape = shape if local is None else (int(local["data_per_step"]), *shape[1:])
            self.eng = Engine(m, prog_shape, cfg, dev, backend=backend)
            self.eng.load_model()
            labels = true["labels"] if local is None else local["labels"][0]
            self.eng.load_targets([g.to(dev) for g in shared[0]["gradients"]], labels.to(dev), mean=meta.mean, std=meta.std)
            if local is not None:
                self.eng.set_local_steps(shape[0], int(local["steps"]), float(local["lr"]), local["labels"])
            x0 = torch.randn(shape, device=dev)
            self.eng.begin_trial(x0, table)
            self.n_params = sum(p.numel() for p in model.parameters())
        self.prog = self.eng.prog

    def warm(self, n):
        self.eng.run(n)
        self.eng.sync()

    def timed(self, n):
        return self.eng.run_timed(n)

    def outputs(self):
        """What a caller of the trial reads back after the last step: the current and the best-so-far candidate, the objective of
        every recorded iteration (warm-up and timed) and, for the joint text attack, the current and best label logits."""
        eng = self.eng
        recorded = eng.status()["recorded"]
        out = dict(candidate=eng.candidate(), best=eng.best(), objective_history=eng.history(min(recorded, self.history_cap)))
        if self.config == 5:
            out.update(labels=eng.joint_labels(best=False), best_labels=eng.joint_labels(best=True))
        return out


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(outputs, directory):
    """Write every output as ``directory/<name>.npy`` (float32).  The largest configuration (5) writes about 13 MB."""
    import numpy as np

    arrays = {name: t.detach().cpu().numpy().astype(np.float32) for name, t in outputs.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"bench.py: outputs of {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte dump limit")
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def host_payload(case, config):
    """The attack inputs as a caller holds them: pinned host tensors (server payload + shared update)."""
    model, loss_fn, payload, shared, true, cfg = case
    pin = lambda t: t.detach().clone().pin_memory()  # noqa: E731
    bufs = payload[0]["buffers"]
    payload_host = [dict(parameters=[pin(p) for p in payload[0]["parameters"]], buffers=None if bufs is None else [pin(b) for b in bufs],
                         metadata=payload[0]["metadata"])]
    meta = dict(shared[0]["metadata"])
    sbufs = shared[0]["buffers"]
    shared_host = [dict(gradients=[pin(g) for g in shared[0]["gradients"]], buffers=None if sbufs is None else [pin(b) for b in sbufs], metadata=meta)]
    h2d = sum(t.numel() * t.element_size() for t in payload_host[0]["parameters"] + (payload_host[0]["buffers"] or [])
              + shared_host[0]["gradients"] + (shared_host[0]["buffers"] or []))
    return payload_host, shared_host, h2d


def product_arm(args):
    import torch
    import torch.distributed as dist

    from breaching_b200 import build as bbuild
    from breaching_b200.attacks import prepare_attack

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product arm has no CPU fallback")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")  # (its banner goes to stderr either way, see _claim_stdout)
        dist.init_process_group("nccl", device_id=dev)
    bbuild.build()
    config = args.config
    w = WORKLOADS[config]
    case = build_case(config)
    model, loss_fn, payload, shared, true, cfg = case
    os.environ["BRE_GEMM_BACKEND"] = args.backend  # also picked up by the attacker of the e2e leg

    runner = EngineRunner(config, case, dev, args.backend, rank)
    warmup = max(args.warmup, 3)
    runner.warm(warmup)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    barrier()
    with ClockSampler(local_rank) as clocks:
        ms = runner.timed(args.steps)
        barrier()
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    if args.dump_outputs and rank == 0:
        dump_outputs(runner.outputs(), args.dump_outputs)
    st = runner.eng.status()
    launches = runner.eng.launches_per_iteration()
    prog, n_params, local_steps = runner.prog, runner.n_params, runner.local_steps
    runner.eng.close()

    # ---- end to end through the public API with HOST (pinned) buffers; N ranks = N restarts, trial k on rank k ------------------
    e2e_steps = args.e2e_steps if args.e2e_steps > 0 else w["e2e_steps"]
    cfg_e2e = copy.deepcopy(cfg)
    cfg_e2e.optim.max_iterations = e2e_steps
    cfg_e2e.optim.callback = e2e_steps
    cfg_e2e.restarts.num_trials = world
    payload_host, shared_host, h2d = host_payload(case, config)
    attacker = prepare_attack(model, loss_fn, cfg_e2e, dict(device=dev, dtype=torch.float))
    barrier()
    t0 = time.perf_counter()
    rec, stats = attacker.reconstruct(payload_host, shared_host, {}, dryrun=False)
    result_host = (rec["raw_embeddings"] if "raw_embeddings" in rec else rec["data"]).to("cpu")
    torch.cuda.synchronize(dev)
    dt = time.perf_counter() - t0
    mine = [k for k in range(world) if k % world == rank]
    executed = sum(len(stats[f"Trial_{k}_Val"]) for k in mine)
    assert all(len(stats[f"Trial_{k}_Val"]) == e2e_steps for k in mine), "a trial of the e2e leg did not run all its iterations"
    counts = torch.tensor([dt, float(executed), float(getattr(attacker, "last_select_seconds", 0.0))], device=dev, dtype=torch.float64)
    if world > 1:
        gathered = [torch.zeros_like(counts) for _ in range(world)]
        dist.all_gather(gathered, counts)
    else:
        gathered = [counts]
    e2e_dt = max(float(g[0]) for g in gathered)
    e2e_iters = sum(float(g[1]) for g in gathered)          # iterations actually executed, summed over ranks
    select_s = max(float(g[2]) for g in gathered)
    d2h = result_host.numel() * result_host.element_size() + executed * 4

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = measured_peaks()
    its = world * args.steps / (ms_max * 1e-3)
    flops_iter = algorithmic_flops(prog, local_steps)
    fam = gemm_family_roofline(dev, prog, args.backend, local_steps)
    peak = peaks["bf16_tflops_sustained"]
    roof = dict(bound="tensor", achieved=fam["tflops"], peak=peak, unit="TFLOP/s", frac=fam["tflops"] / peak,
                traffic=2059008 if config == 2 else None, peak_source=peaks["source"],
                kernel="igemm_tc_kernel (tcgen05 kind::tf32) + SIMT kernels for the shapes it does not cover",
                launches_per_step=fam["n_launches"], avg_launch_us=1e3 * fam["ms_per_launch"], algorithmic_gflop_per_step=fam["flops"] / 1e9,
                peak_tf32_equivalent=peak / 2, frac_of_tf32_peak=fam["tflops"] / (peak / 2), share_of_step=fam["ms_total"] / (ms_max / args.steps),
                whole_step_tflops=flops_iter * (args.steps / (ms_max * 1e-3)) / 1e12,
                note="achieved = algorithmic conv+linear FLOPs of one iteration (SURVEY 8d) / live CUDA-event time of exactly those GEMM "
                     "launches (one graph replay through the C ABI); peak = the measured sustained bf16 cuBLAS rate (the only measured "
                     "tensor peak; the work is TF32, whose dense peak is half of it -> frac_of_tf32_peak); traffic = dram bytes of one "
                     "captured launch (the batch-1 layer2 tangent GEMM, profiles/r2_tc_fprop_dual_b1_summary.txt: = its algorithmic operand bytes)")
    match = matching_reduction_roofline(dev, n_params)
    threads, sweep = cpu_thread_sweep(config, case)
    cpu_its, cpu_dt = oracle_iters_per_sec(config, case, "cpu", 1, args.cpu_steps if args.cpu_steps > 0 else w["ref_steps"])
    eager = None
    if not args.skip_eager and config in (1, 2):
        try:
            eager_its, _ = oracle_iters_per_sec(config, case, dev, 50, args.eager_steps)
            eager = {"value": eager_its, "unit": "it/s", "steps": args.eager_steps, "warmup": 50,
                     "what": "the reference loop (oracle/restate.py = same torch ops as the reference) in eager PyTorch on the same B200, "
                             "cudnn.benchmark on, TF32 convolutions (torch default); denominator of the north-star >=10x target"}
        except Exception as exc:  # noqa: BLE001
            eager = {"value": None, "error": str(exc)}
    out = {
        "metric": w["metric"], "value": its, "unit": "it/s", "n_gpus": world, "steps": args.steps, "warmup": warmup,
        "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "tf32" if args.backend == "tc" else "f32",
        "data": "synthetic",
        "config": {"workload": w["name"] + ", one trial per GPU", "baseline_config": config,
                   "parallelism": f"restarts x{world} (no data-path collective; NCCL MIN select + broadcast once per reconstruct)",
                   "gemm_backend": args.backend, "arithmetic": "fp32 storage; TF32 tensor-core products with fp32 accumulation (= cuDNN's default "
                   "for the reference on a GPU)" if args.backend == "tc" else "fp32",
                   "l2": "per-iteration working set (4+ parameter-sized arenas + activations) exceeds the 126 MB L2 for the 224x224 "
                         "configurations; no explicit flush"},
        "e2e": {"value": e2e_iters / e2e_dt, "unit": "it/s", "h2d_bytes_per_step": world * h2d / e2e_iters, "d2h_bytes_per_step": world * d2h / e2e_iters,
                "steps": e2e_steps, "trials": world, "iterations_executed": e2e_iters, "seconds": e2e_dt, "select_seconds": select_s,
                "phase_seconds_rank0": {k: round(float(v), 4) for k, v in getattr(attacker, "last_timing", {}).items()},
                "what": "prepare_attack(...).reconstruct(host payload, host shared_data) with restarts.num_trials = n_gpus: model rebuild, "
                        "program compile, engine create, H2D of parameters+gradients from pinned memory, every rank runs its own trial for "
                        "all iterations, scoring, cross-rank MIN select + broadcast of the winner (select_seconds), D2H of the result; value "
                        "= iterations actually executed over all ranks / max-over-ranks wall time"},
        "gpu_launches": launches * args.steps, "launches_per_step": launches,
        "clocks": clocks.summary(),
        "roofline": roof,
        "roofline_matching_reduction": match,
        "cpu_baseline": {"value": cpu_its, "unit": "it/s", "cores": threads, "kind": "port",
                         "sample": f"{args.cpu_steps if args.cpu_steps > 0 else w['ref_steps']} iterations of the same workload after 1 warm-up "
                                   f"({cpu_dt:.1f} s), torch CPU ops; thread sweep {sweep} it/s -> {threads} threads (host has {os.cpu_count()} logical CPUs)"},
        "torch_eager_gpu_baseline": eager,
        "final_objective": st["min_objective"],
    }
    _emit(out)
    if world > 1:
        dist.destroy_process_group()


def reference_arm(args):
    """The reference's own CPU implementation of the path = oracle port (the reference is Python and cannot travel to
    the GPU box; oracle/restate.py runs the same torch CPU ops in the same order and is pinned to it by tests/golden)."""
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if rank != 0:
        return
    config = args.config
    w = WORKLOADS[config]
    case = build_case(config)
    threads, sweep = cpu_thread_sweep(config, case)
    its, dt = oracle_iters_per_sec(config, case, "cpu", max(args.warmup, 1), args.steps)
    out = {
        "impl": "reference", "metric": w["metric"], "value": its,
        "unit": "it/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": w["name"], "baseline_config": config, "parallelism": f"host CPU, {threads} threads"},
        "cpu_baseline": {"value": its, "unit": "it/s", "cores": threads, "kind": "port",
                         "sample": f"{args.steps} iterations (one step = one full iteration of the reference loop); thread sweep {sweep} it/s -> "
                                   f"{threads} threads (host has {os.cpu_count()} logical CPUs)"},
        "e2e": {"value": its, "unit": "it/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    _emit(out)


_JSON_OUT = None


def _claim_stdout():
    """The contract is exactly ONE JSON line on rank 0's stdout.  Libraries write there too (NCCL prints its version banner
    from C at NCCL_DEBUG >= VERSION, which the launch environment may set): keep a private handle on the real stdout for the
    result line and point file descriptor 1 at stderr for everything else."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def _emit(obj):
    _JSON_OUT.write(json.dumps(obj) + "\n")
    _JSON_OUT.flush()


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--config", type=int, default=2, choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--backend", default="tc", choices=["simt", "tc"])
    ap.add_argument("--e2e-steps", type=int, default=0)
    ap.add_argument("--cpu-steps", type=int, default=0)
    ap.add_argument("--eager-steps", type=int, default=200)
    ap.add_argument("--skip-eager", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the trial's outputs (rank 0) as DIR/<name>.npy, to compare two builds")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the product arm")
    if args.impl == "reference":
        args.steps = WORKLOADS[args.config]["ref_steps"] if args.steps is None else args.steps
        args.warmup = 3 if args.warmup is None else args.warmup
        if args.config in (3, 4):
            args.warmup = min(args.warmup, 1)
        reference_arm(args)
    else:
        args.steps = (500 if args.config in (1, 2) else 100) if args.steps is None else args.steps
        args.warmup = 50 if args.warmup is None else args.warmup
        product_arm(args)


if __name__ == "__main__":
    main()
