"""The engine's four-sweep formulation (oracle/program_interp.py) equals autograd's double backward (float64)."""
import pytest
import torch

from breaching_b200 import compiler, config, synthetic
from oracle import program_interp as PI
from oracle import restate
from helpers import parity_model

KINDS = ["cosine-similarity", "euclidean", "l1", "tag-euclidean", "angular", "fast-cosine-similarity",
         "masked-cosine-similarity"]


def _setup(mname, data, size, batch, kind, treg=0.0, regs=None):
    H, W = (size, size) if isinstance(size, int) else size
    if mname in ("odd", "tensor-core"):   # the test models of tests/test_sweep_tensors_gpu.py, at their ragged sizes
        model = parity_model(mname, seed=3)
        gen = torch.Generator().manual_seed(4)
        xt = torch.randn(batch, 3, H, W, generator=gen)
        labels = torch.randint(0, model.fc.out_features, (batch,), generator=gen)
        loss_fn = torch.nn.CrossEntropyLoss()
        grads = torch.autograd.grad(loss_fn(model(xt), labels), list(model.parameters()))
        shared, true = [dict(gradients=grads)], dict(labels=labels)
    else:
        model, loss_fn, payload, shared, true = synthetic.make_case(mname, data, batch=batch, seed=3, bn_random=True,
                                                                    image_size=size, classes=10)
    model = model.double().eval()
    g = [t.double() for t in shared[0]["gradients"]]
    gen = torch.Generator().manual_seed(5)
    x = torch.randn(batch, 3, H, W, dtype=torch.double, generator=gen)
    cfg = config.get_attack_config("invertinggradients", {"objective.type": kind, "objective.task_regularization": treg,
                                                           "regularization": regs})
    dm, ds = torch.zeros(1, 3, 1, 1), torch.ones(1, 3, 1, 1)
    orc = restate.TrialOracle(model, loss_fn, cfg, g, true["labels"], dm, ds, dtype=torch.double)
    return model, g, x, true["labels"], cfg, orc


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("mname,data,size", [("convnet-tiny", "cifar", 32), ("resnet18", "imagenet", 32), ("odd", None, (15, 13)),
                                             ("tensor-core", None, (33, 29))])
def test_tangent_formulation_matches_double_backward(mname, data, size, kind):
    model, g, x, labels, cfg, orc = _setup(mname, data, size, 2, kind, treg=0.3)
    phi, _, raw, _ = orc.closure_gradient(x, 0, 0.1)
    prog = compiler.compile_model(model, x.shape)
    it = PI.ProgramInterpreter(model, prog)
    val, dx, loss, G = it.matching_gradient(x, labels, g, kind, scale=1.0, task_regularization=0.3)
    assert abs(float(val) - float(phi)) < 1e-10 * max(1.0, abs(float(phi)))
    assert ((dx - raw).norm() / raw.norm()).item() < 1e-10
    Gref, _ = orc.param_gradient(x, False)
    for a, b in zip(G, Gref):
        assert (a - b).abs().max().item() <= 1e-10 * (b.abs().max().item() + 1e-30)


def test_bottleneck_resnet50():
    model, g, x, labels, cfg, orc = _setup("resnet50", "imagenet", 32, 2, "cosine-similarity")
    phi, _, raw, _ = orc.closure_gradient(x, 0, 0.1)
    it = PI.ProgramInterpreter(model, compiler.compile_model(model, x.shape))
    val, dx, _, _ = it.matching_gradient(x, labels, g, "cosine-similarity")
    assert ((dx - raw).norm() / raw.norm()).item() < 1e-10


def test_regulariser_adjoints_are_injected_into_the_tangent_backward_stream():
    regs = dict(deep_inversion=dict(scale=0.05), features=dict(scale=0.1))
    model, g, x, labels, cfg, orc = _setup("resnet18", "imagenet", 32, 2, "euclidean", regs=regs)
    phi, _, raw, terms = orc.closure_gradient(x, 0, 0.1)
    it = PI.ProgramInterpreter(model, compiler.compile_model(model, x.shape))
    measured = orc._measured.double()
    vals = {}

    def inject(interp):
        v1, inj1 = interp.deep_inversion(0.05, 10)
        v2, inj2 = interp.feature_regularization(measured, 0.1)
        vals["di"], vals["feat"] = float(v1), float(v2)
        out = dict(inj1)
        for k, v in inj2.items():
            out[k] = out.get(k, 0) + v
        return out

    val, dx, _, _ = it.matching_gradient(x, labels, g, "euclidean", inject_fn=inject)
    assert abs(vals["di"] - terms["deep_inversion"]) < 1e-9 * max(1.0, abs(terms["deep_inversion"]))
    assert abs(vals["feat"] - terms["features"]) < 1e-9 * max(1.0, abs(terms["features"]))
    assert ((dx - raw).norm() / raw.norm()).item() < 1e-9


@pytest.mark.parametrize("mname,data,size,batch", [("convnet-tiny", "cifar", 32, 3), ("resnet18", "imagenet", 32, 2)])
def test_train_mode_batchnorm_rules_match_double_backward(mname, data, size, batch):
    """No server / user buffers (base_attack.py:192-197): the attacked model runs BatchNorm in train mode with
    ``track_running_stats = False`` -- batch statistics of the candidate itself, so every BN couples the whole batch in the
    forward, the backward and both tangent sweeps."""
    model, g, x, labels, cfg, orc = _setup(mname, data, size, batch, "cosine-similarity", treg=0.2)
    model.train()
    for mod in model.modules():
        if hasattr(mod, "track_running_stats"):
            mod.track_running_stats = False
    phi, _, raw, _ = orc.closure_gradient(x, 0, 0.1)
    prog = compiler.compile_model(model, x.shape)
    assert any(getattr(op, "bn_train", False) for op in prog.ops)
    it = PI.ProgramInterpreter(model, prog)
    val, dx, loss, G = it.matching_gradient(x, labels, g, "cosine-similarity", scale=1.0, task_regularization=0.2)
    assert abs(float(val) - float(phi)) < 1e-9 * max(1.0, abs(float(phi)))
    assert ((dx - raw).norm() / raw.norm()).item() < 1e-8
    Gref, _ = orc.param_gradient(x, False)
    scale = max(b.abs().max().item() for b in Gref)   # conv biases in front of a train-mode BN have an exactly-zero gradient
    for a, b in zip(G, Gref):
        assert (a - b).abs().max().item() <= 1e-9 * b.abs().max().item() + 1e-12 * scale
