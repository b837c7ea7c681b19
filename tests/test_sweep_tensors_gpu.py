"""Every intermediate buffer of the engine's four sweeps against the float64 layer program (oracle/program_interp.py).

One closure evaluation per case; then, for every tensor id, what sweep F wrote (``val``), sweep B (``delta``), sweep TF (``tangent``)
and sweep TB (``tangent_delta``), and every parameter gradient G (and, on the fp32 back end, the direction v), each against the
interpreter's ``a`` / ``d_B`` / ``ta`` / ``d_TB`` / ``G`` / ``v`` by relative l2 error.  The cases are small models that reach
dispatch branches the end-to-end tests do not; the engine switches (environment variables, read once per process) run in child
processes, the engine options in-process.

Measured worst per-tensor error (NVIDIA B200, 1000 W power limit; the bounds in TOL are about 3x these):

    case          simt      tc        worst tensor on tc
    odd           4.9e-6    3.8e-6    (no tensor-core layer)
    odd_train     3.3e-4    3.0e-4    G of the conv biases in front of a train-mode BN (exactly zero in float64), with a floor
                                      of 1e-4; 3.3e-5 with the floor of 1e-3 used now
    tcnet         5.7e-5    5.6e-2    tangent of the stride-2 block's BN output
    resnet18_di   1.3e-6    8.1e-2    tangent of a layer2 conv output
    text          5.0e-7    1.6e-3    G of the QKV projection

Every scheduling switch left every buffer bit-identical.  FedAvg (tc): rel(fused, simt) = rel(unfused, simt) = 4.6e-4 (ConvNet)
and 0.235 (ResNet-18).
"""
import argparse
import copy
import functools
import os
import subprocess
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for _p in (ROOT, HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from breaching_b200 import compiler, config, synthetic  # noqa: E402
from helpers import FEDAVG_FIXTURES, case_from_fixture, cfg_from_fixture, load_golden, parity_model  # noqa: E402
from oracle import program_interp as PI  # noqa: E402

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
SWEEPS = ("val", "delta", "tangent", "tangent_delta")
KIND = "cosine-similarity"
DI_SCALE = 0.05
_PDL_DEFAULT = os.environ.get("BRE_PDL", "1").strip() not in ("0", "")   # what the engine reads when no option overrides it

# Cases and the branches each one reaches:
#   odd          OddChannelNet (3 -> 6 -> 10 -> 14), eval BN with random running statistics, residual add, 3/2/1 max-pool on 15 x 13,
#                average pool, 7 classes, batch 3: the scalar bnact / pool / channel-statistics kernels (no channel count is a
#                multiple of 4), acc_in accumulation of the residual operand's deltas, SIMT GEMMs on both back ends
#   odd_train    the same topology with train-mode BN (no running statistics): bn_train_* kernels on odd channel counts
#   tcnet        TensorCoreNet on 33 x 29, batch 2: the stem column path (stem_cols.cu), 128 x 32 tiles (32 / 96 channels) and
#                128 x 64 tiles, per-parity-class strided dgrad (3 x 3 and 1 x 1 stride 2), ragged M tiles, split-K clusters
#   resnet18_di  ResNet-18 at 64 x 64, batch 2, DeepInversion prior: max-pool after ReLU, downsample accumulation, batched DI
#                statistics and the DI adjoint inside sweep TB
#   text         transformer (ninp 32, 8192-token vocabulary, soft labels), batch 2 x 8 tokens: linear_tall decoder dgrad, 128 x 32
#                tiles of the 96-wide QKV projection, the token kernels inside a full program
CASES = ["odd", "odd_train", "tcnet", "resnet18_di", "text"]

# per-tensor bound on the relative l2 error: about 3x the measured worst (module docstring).  On "tc" the TF32 operands (10-bit
# mantissa) of every GEMM compound through the forward, backward and both tangent sweeps: the tangents and tangent deltas of the
# 64- and 128-channel layers end 5-8 % from float64 -- the same order as the TF32 tolerances of the end-to-end tests (5 % on the
# candidate gradient in smoke(), 27 % for FedAvg).  A buffer the engine fails to write is 100 % off.
TOL = {
    ("odd", "simt"): 1.5e-5, ("odd", "tc"): 1.5e-5,   # no layer of this net runs on the tensor cores
    ("odd_train", "simt"): 1e-4, ("odd_train", "tc"): 1e-4,
    ("tcnet", "simt"): 2e-4, ("tcnet", "tc"): 0.17,
    ("resnet18_di", "simt"): 4e-6, ("resnet18_di", "tc"): 0.25,
    ("text", "simt"): 1.5e-6, ("text", "tc"): 5e-3,
}
# a tensor is compared relative to max(its own norm, FLOOR x the largest norm of the same sweep): the conv biases in front of a
# train-mode BN have an exactly-zero gradient, which no fp32 sum reproduces
FLOOR = 1e-3


# ---------------------------------------------------------------------------------------------------------------- cases
def _cfg(di=False):
    regs = dict(deep_inversion=dict(scale=DI_SCALE)) if di else None
    return config.get_attack_config("invertinggradients", {"objective.type": KIND, "objective.task_regularization": 0.0,
                                                            "regularization": regs})


def _vision(model, shape, seed):
    gen = torch.Generator().manual_seed(seed)
    classes = model.fc.out_features
    xt, x = torch.randn(shape, generator=gen), torch.randn(shape, generator=gen)
    labels = torch.randint(0, classes, (shape[0],), generator=gen)
    grads = torch.autograd.grad(torch.nn.functional.cross_entropy(model(xt), labels), list(model.parameters()))
    return dict(model=model, shape=shape, x=x, labels=labels, g=[t.detach() for t in grads], program=None, soft=None)


@functools.lru_cache(maxsize=None)
def make_case(name):
    if name in ("odd", "odd_train"):
        c = _vision(parity_model("odd", seed=11, train_bn=name == "odd_train"), (3, 3, 15, 13), 12)
    elif name == "tcnet":
        c = _vision(parity_model("tensor-core", seed=13), (2, 3, 33, 29), 14)
    elif name == "resnet18_di":
        model = synthetic.build_model("resnet18", 10, seed=15)
        synthetic.randomize_bn(model, 16)
        c = _vision(model.eval(), (2, 3, 64, 64), 17)
    elif name == "text":
        model, loss_fn, payload, shared, true = synthetic.make_text_case(batch=2, seq_len=8, seed=19, ntokens=8192, ninp=32, nhead=4,
                                                                          nhid=64, nlayers=1)
        names = [n for n, _ in model.named_parameters()]
        g = list(shared[0]["gradients"])
        g.pop(names.index("encoder.weight"))
        gen = torch.Generator().manual_seed(20)
        B, T, d, V = 2, 8, 32, 8192
        c = dict(model=model, shape=(B * T, d, 1, 1), x=torch.randn(B, T, d, generator=gen), labels=torch.zeros(B * T, dtype=torch.long),
                 g=g, program=compiler.compile_transformer(model, B, T), soft=torch.randn(B, T, V, generator=gen).softmax(dim=-1))
        assert c["program"].logits_valid in (0, V)   # no padded vocabulary: the interpreter runs the same program
    else:
        raise KeyError(name)
    c["cfg"] = _cfg(di=name == "resnet18_di")
    c["di"] = name == "resnet18_di"
    return c


class _TokenParams:   # parameters in program order (the token embedding is not part of the attacked program)
    def __init__(self, model):
        self.model = model

    def parameters(self):
        return [p for n, p in self.model.named_parameters() if n != "encoder.weight"]

    def named_modules(self):
        return self.model.named_modules()


@functools.lru_cache(maxsize=None)
def reference(name):
    """float64 buffers of the four sweeps, keyed like :func:`read_buffers`."""
    c = make_case(name)
    m64 = copy.deepcopy(c["model"]).double()
    if c["program"] is not None:
        prog = compiler.compile_transformer(c["model"], 2, 8, pad_vocab=False)
        it = PI.ProgramInterpreter(_TokenParams(m64), prog)
        targets = c["soft"].double()
    else:
        prog = compiler.compile_model(m64, c["shape"])
        it = PI.ProgramInterpreter(m64, prog)
        targets = c["labels"]
    g64 = [t.double() for t in c["g"]]
    inject = {}

    def di(interp):
        inject.update(interp.deep_inversion(DI_SCALE, 10)[1])
        return inject

    _, dx, _, G = it.matching_gradient(c["x"].double(), targets, g64, KIND, inject_fn=di if c["di"] else None)
    _, V = PI.objective_direction(KIND, G, g64)
    ref = {("grad", 0): dx}
    for tid in range(len(prog.tensors)):
        ref[("val", tid)] = it.a[tid]
        ref[("tangent_delta", tid)] = it.d_TB[tid] + inject.get(tid, 0)   # the engine adds the DI adjoint where BN reads its input
        if tid != 0:   # the candidate has no tangent, and no delta without a task-loss term
            ref[("delta", tid)] = it.d_B[tid]
            ref[("tangent", tid)] = it.ta[tid]
    for i, (gi, vi) in enumerate(zip(G, V)):
        ref[("G", i)], ref[("v", i)] = gi, vi
    return ref, prog


# ---------------------------------------------------------------------------------------------------------------- engine side
def run_engine(name, backend, options=()):
    """One closure evaluation on a fresh engine with ``options`` applied; returns the engine and its returned gradient."""
    from breaching_b200.engine import Engine

    c = make_case(name)
    dev = torch.device(DEV)
    model = None if c["program"] is not None else copy.deepcopy(c["model"]).to(dev)
    eng = Engine(model, c["shape"], c["cfg"], dev, backend=backend, program=c["program"])
    for key, value in options:
        eng.set_option(key, value)
    if c["program"] is not None:
        eng.load_model(params=[p.detach() for p in _TokenParams(c["model"]).parameters()])
    else:
        eng.load_model()
    eng.load_targets([t.to(dev) for t in c["g"]], c["labels"].to(dev))
    if c["soft"] is not None:
        eng.load_soft_labels(c["soft"].reshape(c["shape"][0], -1).to(dev))
    _, grad = eng.objective_and_gradient(c["x"].reshape(c["shape"]).to(dev))
    return eng, grad


def read_buffers(eng, grad, x):
    out = {("grad", 0): grad.cpu()}
    for tid in range(len(eng.prog.tensors)):
        for sweep in SWEEPS:
            if tid == 0 and sweep == "tangent":
                continue
            out[(sweep, tid)] = eng.debug_tensor(sweep, tid)
    for i in range(len(eng.prog.params)):
        out[("G", i)] = eng.debug_param("G", i)
        out[("v", i)] = eng.debug_param("v", i)
    # launch count of one optimiser iteration (the captured iteration counts its launches; the closure call alone does not)
    eng.begin_trial(x, [0.0])
    eng.run(1)
    eng.sync()
    out[("launches", 0)] = torch.tensor([eng.launches_per_iteration()])
    return out


def engine_buffers(name, backend, options=()):
    eng, grad = run_engine(name, backend, options)
    try:
        c = make_case(name)
        return read_buffers(eng, grad, c["x"].reshape(c["shape"]).to(DEV))
    finally:
        if any(k == "pdl" for k, _ in options):   # process-global: restore it for every later engine
            eng.set_option("pdl", int(_PDL_DEFAULT))
        eng.close()


# ---------------------------------------------------------------------------------------------------------------- comparison
def _producer(prog, tid):
    for i, op in enumerate(prog.ops):
        if op.tout == tid:
            return i, compiler.OP_NAMES[op.kind]
    return -1, "candidate"


def compare(name, backend, got, fused=False):
    """Per-tensor relative l2 errors against float64.  Returns (records sorted worst first, skipped keys).

    Skipped: ``v`` on the tensor-core back end (make_v writes only the TF32 shadow of tensor-core weights there), the candidate's
    delta (no task-loss term), and -- with ``fused`` -- the pre-BN tangents the fused epilogue does not store (a conv output whose
    only consumer is the following BN; those read back as the zeros the buffer was allocated with)."""
    ref, prog = reference(name)
    pool_in = {op.tin for op in prog.ops if op.kind == compiler.OP_MAXPOOL}
    one_reader = {op.tout for i, op in enumerate(prog.ops)
                  if op.kind == compiler.OP_CONV and i + 1 < len(prog.ops) and prog.ops[i + 1].kind == compiler.OP_BNACT
                  and prog.ops[i + 1].tin == op.tout and sum((o.tin == op.tout) + (o.res == op.tout) for o in prog.ops) == 1}
    scale = {}
    for (sweep, idx), r in ref.items():
        scale[sweep] = max(scale.get(sweep, 0.0), float(r.norm()))
    records, skipped = [], []
    for key, r in ref.items():
        sweep, idx = key
        if sweep == "v" and backend == "tc":
            continue
        if sweep == "delta" and idx == 0:
            continue
        e = got[key].double().reshape(r.shape)
        if fused and sweep == "tangent" and idx in one_reader and not bool(e.any()):
            skipped.append(key)
            continue
        if sweep in ("delta", "tangent_delta") and idx in pool_in:
            # max-pool ties after a ReLU: a window of zeros sends its delta to another zero than torch does; the ReLU in front masks
            # those positions anyway
            keep = (ref[("val", idx)] > 0).to(r.dtype)
            e, r = e * keep, r * keep
        if not bool(torch.isfinite(e).all()):
            err = float("inf")
        else:
            err = float((e - r).norm() / max(float(r.norm()), FLOOR * scale[sweep], 1e-300))
        if sweep in ("G", "v"):
            where = f"param {idx} {tuple(r.shape)}"
        else:
            op_i, kind = _producer(prog, idx)
            where = f"tensor {idx} (op {op_i} {kind}) {tuple(r.shape)}"
        records.append((err, sweep, where))
    records.sort(key=lambda t: -t[0])
    return records, skipped


def _worst(records, n=3):
    return "; ".join(f"{s} {w}: {e:.3e}" for e, s, w in records[:n])


def _differs(a, b):
    """Keys whose buffers are not bit-identical."""
    return sorted(k for k in a if k in b and not torch.equal(a[k], b[k]))


# ---------------------------------------------------------------------------------------------------------------- 1. parity
@pytest.mark.parametrize("backend", ["simt", "tc"])
@pytest.mark.parametrize("name", CASES)
def test_sweep_tensors_match_float64(name, backend):
    got = engine_buffers(name, backend)
    records, skipped = compare(name, backend, got)
    assert not skipped
    tol = TOL[(name, backend)]
    print(f"\nMEASURED {name} {backend}: worst {records[0][0]:.3e} ({_worst(records, 1)})")
    assert records[0][0] < tol, f"{name}/{backend}: worst per-tensor errors {_worst(records)} (bound {tol:.1e})"


# ---------------------------------------------------------------------------------------------------------------- 2. options
# (options, must be bit-identical to the default).  precise_last=2: the last GEMM of both nets is a 10-class head that runs on the
# fp32 kernel anyway (precise_last=1 changes nothing there); the second-last is a tensor-core convolution.
OPTIONS = {
    "pdl0": ((("pdl", 0),), True),
    "overlap_wgrad0": ((("overlap_wgrad", 0),), True),
    "fuse_bnact": ((("fuse_bnact", 1),), False),
    "precise_first2": ((("precise_first", 2),), False),
    "precise_last2": ((("precise_last", 2),), False),
    "fuse_precise_first2": ((("fuse_bnact", 1), ("precise_first", 2)), False),
    "fuse_precise_last2": ((("fuse_bnact", 1), ("precise_last", 2)), False),
}


@functools.lru_cache(maxsize=None)
def _default_tc(name):
    return engine_buffers(name, "tc")


@pytest.mark.parametrize("option", list(OPTIONS))
@pytest.mark.parametrize("name", ["tcnet", "resnet18_di"])
def test_engine_options(name, option):
    opts, identical = OPTIONS[option]
    base = _default_tc(name)
    got = engine_buffers(name, "tc", opts)
    _check_setting(name, got, base, identical, fused=any(k == "fuse_bnact" for k, _ in opts), label=option)


def _check_setting(key, got, base, identical, fused=False, label="", loose=None):
    name, backend = (key.split(":") + ["tc"])[:2]
    diff = _differs(got, base)
    if identical:
        assert not diff, f"{label} on {name}: not bit-identical to the default run in {diff[:6]}"
        return
    assert diff, f"{label} on {name}: nothing changed, so the case does not reach its branch"
    records, skipped = compare(name, backend, got, fused=fused)
    if fused:
        assert skipped, "fuse_bnact fused no layer"
    assert all(k[0] == "tangent" for k in skipped)
    bound = TOL[(name, backend)] if loose is None else loose
    assert records[0][0] < bound, f"{label} on {name}: worst per-tensor errors {_worst(records)} (bound {bound:.2e})"


# ---------------------------------------------------------------------------------------------------------------- 2. environment
SCHEDULING = ["BRE_PDL=0", "BRE_TC_WPREFETCH=0", "BRE_TC_PRODUCERS=1", "BRE_TC_PRODUCERS=3", "BRE_TC_PRODUCERS=4", "BRE_TC_STAGES=2",
              "BRE_TC_STAGES=8", "BRE_TC_SHORTK_STAGES=4"]
KERNELS = ["BRE_VEC_EW=0", "BRE_DEFER_BN=0", "BRE_DI_BATCHED=0", "BRE_STEM_COLS=0", "BRE_TC_TMA=0", "BRE_TC_STRIDED_TMA=0",
           "BRE_TC_NARROW=0", "BRE_TC_MAX_SPLITS=1", "BRE_TC_TARGET_CTAS=4096", "BRE_TC_ROUND=0"]
TEXT_KERNELS = ["BRE_LINEAR_SMALL=0", "BRE_LINEAR_SMALL_ROWS=1", "BRE_LINEAR_TALL=0"]
MATRIX_CASES = ["tcnet:tc", "resnet18_di:tc"]
TEXT_CASES = ["text:tc", "text:simt"]   # BRE_LINEAR_SMALL selects a kernel of the fp32 back end


def _child(setting, cases, tmp_path):
    """Run this file as a script with exactly one BRE_* variable set; returns {case: buffers}."""
    env = {k: v for k, v in os.environ.items() if not k.startswith("BRE_")}
    if setting:
        k, v = setting.split("=")
        env[k] = v
    out = tmp_path / (setting.replace("=", "_") or "default")
    out.mkdir(exist_ok=True)
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), "--out", str(out), "--cases",
                                                                         ",".join(cases)]
    res = subprocess.run(cmd, env=env, timeout=600, capture_output=True, text=True, cwd=ROOT)
    assert res.returncode == 0, f"child with {setting or 'no switch'} failed:\n{res.stdout[-2000:]}\n{res.stderr[-4000:]}"
    return {c: torch.load(out / f"{c.replace(':', '_')}.pt", weights_only=False) for c in cases}


@pytest.fixture(scope="module")
def defaults(tmp_path_factory):
    return _child("", MATRIX_CASES + TEXT_CASES, tmp_path_factory.mktemp("defaults"))


@pytest.mark.parametrize("setting", SCHEDULING)
def test_scheduling_switch_is_bit_identical(setting, defaults, tmp_path):
    got = _child(setting, MATRIX_CASES, tmp_path)
    for key in MATRIX_CASES:
        _check_setting(key, got[key], defaults[key], True, label=setting)


@pytest.mark.parametrize("setting", KERNELS + TEXT_KERNELS)
def test_kernel_switch_meets_the_float64_bound(setting, defaults, tmp_path):
    cases = TEXT_CASES if setting in TEXT_KERNELS else MATRIX_CASES
    got = _child(setting, cases, tmp_path)
    reached = []
    for key in cases:
        name, backend = key.split(":")
        loose = None
        if setting == "BRE_TC_ROUND=0":   # truncated TF32 operands (documented as less accurate): 3x the default's own error
            loose = 3 * compare(name, backend, defaults[key])[0][0][0]
        reached.append(bool(_differs(got[key], defaults[key])))
        if reached[-1]:
            _check_setting(key, got[key], defaults[key], False, label=setting, loose=loose)
    assert any(reached), f"{setting} changed no launch count and no bit on {cases}: no case reaches its branch"


# ---------------------------------------------------------------------------------------------------------------- 3. FedAvg
@pytest.mark.parametrize("name", FEDAVG_FIXTURES)
def test_fedavg_fused_epilogue_is_no_worse_than_unfused(name):
    """FedAvg carries the adjoint back over the local steps with tangent gamma-gradients, which read the pre-BN tangent; the fused
    epilogue must store it then.  Both tensor-core runs against the fp32 run of the same engine."""
    from breaching_b200.engine import Engine

    fx = load_golden(f"trial_{name}.pt")
    model, loss_fn, payload, shared, true = case_from_fixture(fx)
    cfg = cfg_from_fixture(fx)
    local = shared[0]["metadata"]["local_hyperparams"]
    meta = payload[0]["metadata"]
    dev = torch.device(DEV)
    grads = {}
    for label, backend, fuse in (("simt", "simt", 0), ("unfused", "tc", 0), ("fused", "tc", 1)):
        eng = Engine(copy.deepcopy(model).to(dev).eval(), (local["data_per_step"], *fx["x0"].shape[1:]), cfg, dev, backend=backend)
        eng.set_option("fuse_bnact", fuse)
        eng.load_model()
        eng.load_targets([g.to(dev) for g in shared[0]["gradients"]], local["labels"][0], mean=meta.mean, std=meta.std)
        eng.set_local_steps(fx["x0"].shape[0], local["steps"], local["lr"], local["labels"])
        grads[label] = eng.objective_and_gradient(fx["x0"].to(dev))[1].double().cpu()
        eng.close()

    def rel(a, b):
        return float((a - b).norm() / b.norm())

    fused, unfused = rel(grads["fused"], grads["simt"]), rel(grads["unfused"], grads["simt"])
    print(f"\nMEASURED fedavg {name}: rel(fused, simt) {fused:.3e}, rel(unfused, simt) {unfused:.3e}")
    assert fused <= 1.5 * unfused + 1e-4, (fused, unfused)


# ---------------------------------------------------------------------------------------------------------------- child process
def _main():
    ap = argparse.ArgumentParser(description="dump the four-sweep buffers of the given cases (name:backend, comma-separated)")
    ap.add_argument("--out", required=True)
    ap.add_argument("--cases", required=True)
    args = ap.parse_args()
    for key in args.cases.split(","):
        name, backend = key.split(":")
        torch.save(engine_buffers(name, backend), os.path.join(args.out, f"{name}_{backend}.pt"))


if __name__ == "__main__":
    _main()
