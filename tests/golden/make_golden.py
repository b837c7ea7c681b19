"""Generate the golden fixtures in this directory by running the UNMODIFIED reference.

Run in the build container (needs /root/reference):  ``python tests/golden/make_golden.py``

The reference ships no tests or golden vectors for the optimisation hot path (SURVEY.md section 4), so the parity pin
is produced here: the reference attacker (``breaching.attacks.prepare_attack`` imported from /root/reference through
``oracle/refshim.py``) is driven on small seeded synthetic cases and its per-iteration outputs are stored.
``tests/test_golden.py`` checks the oracle restatement against these files on any machine; the ``-m gpu`` tests check
the CUDA engine against them on the B200 box, where /root/reference does not exist.
"""
import copy
import os
import sys
import warnings

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
warnings.filterwarnings("ignore")

from breaching_b200 import synthetic  # noqa: E402
from oracle import refshim  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))

CASES = {
    # name: (case kwargs, attack yaml, overrides, iterations)
    "ig_convnet": (dict(model_name="convnet-tiny", data="cifar", batch=2, seed=3, bn_random=True),
                   "invertinggradients", {}, 8),
    "ig_resnet18": (dict(model_name="resnet18", data="imagenet", batch=1, seed=5, bn_random=True, image_size=64, classes=10),
                    "invertinggradients", {}, 6),
    "stg_resnet18": (dict(model_name="resnet18", data="imagenet", batch=2, seed=11, image_size=64, classes=10,
                          user_buffers=True),
                     "seethroughgradients", {"optim.langevin_noise": 0.0}, 6),
    "modern_convnet": (dict(model_name="convnet-tiny", data="cifar", batch=2, seed=7, bn_random=True),
                       "modern", {"regularization.features.scale": 0.1, "regularization.deep_inversion.scale": 0.01}, 6),
    "tag_clip_convnet": (dict(model_name="convnet-tiny", data="cifar", batch=1, seed=9, bn_random=True),
                         "invertinggradients",
                         {"objective.type": "tag-euclidean", "objective.tag_scale": 0.1, "objective.scale_scheme": "linear",
                          "objective.task_regularization": 0.2, "optim.optimizer": "bert-adam", "optim.signed": None,
                          "optim.grad_clip": 0.5, "optim.step_size_decay": "linear", "optim.warmup": 3,
                          "optim.boxed": False}, 8),
    "l1_sgd_convnet": (dict(model_name="convnet-tiny", data="cifar", batch=1, seed=13, bn_random=True),
                       "invertinggradients",
                       {"objective.type": "l1", "objective.scale": 0.01, "optim.optimizer": "momgd", "optim.signed": "soft",
                        "optim.step_size": 0.01, "optim.step_size_decay": "cosine-decay",
                        "regularization.total_variation.double_opponents": True,
                        "regularization.total_variation.inner_exp": 2, "regularization.total_variation.outer_exp": 0.5}, 6),
}


TRAIN_BN_CASES = {
    # no BN buffers anywhere: the reference puts the attacked model in train mode (base_attack.py:192-197)
    "trainbn_convnet": (dict(model_name="convnet-tiny", data="cifar", batch=3, seed=61, bn_random=True, no_buffers=True),
                        "invertinggradients", {"optim.signed": "soft"}, 6),
    "trainbn_resnet18": (dict(model_name="resnet18", data="imagenet", batch=2, seed=62, bn_random=True, no_buffers=True, image_size=64,
                              classes=10), "invertinggradients", {"optim.signed": "soft"}, 4),
}

LBFGS_CASES = {
    # L-BFGS presets (common.py:18; `beyondinfering.yaml`, `wei.yaml`): 20 inner iterations per optimizer.step, hard-signed
    # gradients (the default `optim.signed`) resp. task-loss regularisation + euclidean matching
    "lbfgs_convnet": (dict(model_name="convnet-tiny", data="cifar", batch=1, seed=15, bn_random=True), "beyondinfering", {}, 3),
    "lbfgs_wei_convnet": (dict(model_name="convnet-tiny", data="cifar", batch=2, seed=16, bn_random=True), "wei",
                          {"optim.signed": None}, 3),
    "lbfgs_cosine_convnet": (dict(model_name="convnet-tiny", data="cifar", batch=2, seed=17, bn_random=True), "invertinggradients",
                             {"optim.optimizer": "L-BFGS", "optim.signed": None, "optim.step_size": 0.5,
                              "optim.step_size_decay": "cosine-decay"}, 4),
}

JOINT_CASES = {
    # attack_type joint-optimization (optimization_with_label_attack.py): data and soft labels optimised together
    "joint_dlg_convnet": (dict(model_name="convnet-tiny", data="cifar", batch=1, seed=21, bn_random=True), "deepleakage", {}, 3),
    "joint_adam_convnet": (dict(model_name="convnet-tiny", data="cifar", batch=2, seed=22, bn_random=True), "invertinggradients",
                           {"attack_type": "joint-optimization", "label_strategy": None, "optim.signed": "soft",
                            "optim.step_size": 0.05, "optim.grad_clip": 0.5}, 6),
    # BASELINE config 5 in miniature: TAG (tag.yaml) on a 2-layer transformer, candidate in embedding space, token-level soft labels
    "joint_tag_transformer": (dict(batch=1, seq_len=8, seed=51, ntokens=50, ninp=16, nhead=4, nhid=24, nlayers=2), "tag",
                              {"optim.warmup": 2}, 6),
}

MULTI_QUERY_CASES = {
    # two model queries answered on the same user batch; the objective sums over them (optimization_based_attack.py:157-160)
    "multiquery_convnet": (dict(model_name="convnet-tiny", data="cifar", batch=2, seed=31, queries=2, bn_random=True),
                           "invertinggradients", {"optim.signed": "soft"}, 6),
}

FEDAVG_CASES = {
    # FedAvg multi-step updates (objectives.py:48-72).  `features` / `deep_inversion` crash in the reference together with
    # FedAvg (SURVEY.md fact 9), so the fixture uses the `modern` preset with the features prior switched off.
    "fedavg_convnet": (dict(model_name="convnet-tiny", data="cifar", num_data_points=4, steps=3, data_per_step=2, lr=0.05, seed=4,
                            bn_random=True), "modern", {"regularization.features.scale": 0.0}, 6),
    "fedavg_resnet18": (dict(model_name="resnet18", data="imagenet", num_data_points=4, steps=4, data_per_step=1, lr=0.01, seed=6,
                             bn_random=True, image_size=64, classes=10), "modern", {"regularization.features.scale": 0.0}, 4),
}


def run_reference(ref, case_kwargs, attack, overrides, iters):
    if "steps" in case_kwargs:
        model, loss_fn, payload, shared, true = synthetic.make_fedavg_case(**case_kwargs)
    elif "queries" in case_kwargs:
        model, loss_fn, payload, shared, true = synthetic.make_multi_query_case(**case_kwargs)
    else:
        model, loss_fn, payload, shared, true = synthetic.make_case(**case_kwargs)
    local_hyperparams = shared[0]["metadata"]["local_hyperparams"]
    cfg = refshim.load_reference_attack_cfg(attack, overrides)
    setup = dict(device=torch.device("cpu"), dtype=torch.float)
    attacker = ref.attacks.prepare_attack(model, loss_fn, cfg, setup)
    shared_ref = copy.deepcopy(shared)
    rec_models, labels, stats = attacker.prepare_attack(payload, shared_ref)
    for r in attacker.regularizers:
        r.initialize(rec_models, shared_ref, labels)
    attacker.objective.initialize(attacker.loss_fn, attacker.cfg.impl, local_hyperparams)
    n = shared[0]["metadata"]["num_data_points"]
    gen = torch.Generator().manual_seed(case_kwargs["seed"] + 1000)
    x0 = torch.randn([n, *attacker.data_shape], generator=gen)

    # (1) raw objective + gradient at x0 through the reference's own closure with post-processing disabled
    cfg_raw = copy.deepcopy(cfg)
    cfg_raw.optim.signed = None
    cfg_raw.optim.grad_clip = None
    cfg_raw.optim.langevin_noise = 0.0
    att_raw = ref.attacks.prepare_attack(model, loss_fn, cfg_raw, setup)
    att_raw.dm, att_raw.ds, att_raw.data_shape = attacker.dm, attacker.ds, attacker.data_shape
    for r in att_raw.regularizers:
        r.initialize(rec_models, shared_ref, labels)
    att_raw.objective.initialize(att_raw.loss_fn, att_raw.cfg.impl, local_hyperparams)
    cand = att_raw._initialize_data([n, *attacker.data_shape])
    cand.data = x0.clone()
    opt_raw, _ = att_raw._init_optimizer([cand])
    obj0 = att_raw._compute_objective(cand, labels, rec_models, opt_raw, shared_ref, 0)()
    raw_grad = cand.grad.detach().clone()
    task_loss0 = float(att_raw.current_task_loss)

    # (2) the reference loop body, iteration by iteration (optimization_based_attack.py:110-121)
    cand = attacker._initialize_data([n, *attacker.data_shape])
    cand.data = x0.clone()
    optimizer, scheduler = attacker._init_optimizer([cand])
    best = cand.detach().clone()
    fmin = torch.as_tensor(float("inf"))
    history, lrs, cands = [], [], []
    for it in range(iters):
        lrs.append(optimizer.param_groups[0]["lr"])
        closure = attacker._compute_objective(cand, labels, rec_models, optimizer, shared_ref, it)
        val = optimizer.step(closure)
        scheduler.step()
        with torch.no_grad():
            if attacker.cfg.optim.boxed:
                cand.data = torch.max(torch.min(cand, (1 - attacker.dm) / attacker.ds), -attacker.dm / attacker.ds)
            if val < fmin:
                fmin = val.detach()
                best = cand.detach().clone()
        history.append(val.item())
        cands.append(cand.detach().clone())
    # (3) scoring of the best candidate with the reference's _score_trial
    score = float(attacker._score_trial(best, labels, rec_models, shared_ref))
    checksum = float(sum(p.double().sum() for p in model.parameters()))
    return dict(
        case=case_kwargs, attack=attack, overrides=overrides, iters=iters, x0=x0, labels=labels, true_labels=true["labels"],
        objective0=float(obj0), task_loss0=task_loss0, raw_grad0=raw_grad, history=history, lrs=lrs,
        candidate_after_1=cands[0], candidate_final=cands[-1], best=best, score=score, scoring=cfg.restarts.scoring,
        weight_checksum=checksum, torch_version=torch.__version__,
    )


def run_reference_joint(ref, case_kwargs, attack, overrides, iters):
    """Drive the reference's OptimizationJointAttacker loop body (optimization_with_label_attack.py:100-128) iteration by
    iteration from seeded initial data / label logits."""
    if "seq_len" in case_kwargs:
        model, loss_fn, payload, shared, true = synthetic.make_text_case(**case_kwargs)
    else:
        model, loss_fn, payload, shared, true = synthetic.make_case(**case_kwargs)
    cfg = refshim.load_reference_attack_cfg(attack, overrides)
    setup = dict(device=torch.device("cpu"), dtype=torch.float)
    attacker = ref.attacks.prepare_attack(model, loss_fn, cfg, setup)
    shared_ref = copy.deepcopy(shared)
    rec_models, label_template, stats = attacker.prepare_attack(payload, shared_ref)
    attacker.objective.initialize(attacker.loss_fn, attacker.cfg.impl, None)
    n = shared[0]["metadata"]["num_data_points"]
    gen = torch.Generator().manual_seed(case_kwargs["seed"] + 1000)
    x0 = torch.randn([n, *attacker.data_shape], generator=gen)
    l0 = torch.randn(list(label_template.shape), generator=gen)
    cand = attacker._initialize_data([n, *attacker.data_shape])
    cand.data = x0.clone()
    labels = attacker._initialize_data(label_template.shape)
    labels.data = l0.clone()
    optimizer, scheduler = attacker._init_optimizer([cand, labels])
    best, best_l, fmin = cand.detach().clone(), labels.detach().clone(), torch.as_tensor(float("inf"))
    history, lrs = [], []
    raw = None
    for it in range(iters):
        lrs.append(optimizer.param_groups[0]["lr"])
        closure = attacker._compute_objective(cand, labels, rec_models, optimizer, shared_ref, it)
        val = optimizer.step(closure)
        scheduler.step()
        with torch.no_grad():
            if attacker.cfg.optim.boxed:
                cand.data = torch.max(torch.min(cand, (1 - attacker.dm) / attacker.ds), -attacker.dm / attacker.ds)
            if val < fmin:
                fmin, best, best_l = val.detach(), cand.detach().clone(), labels.detach().clone()
        history.append(val.item())
    # raw objective and gradients at the initial point (post-processing disabled)
    cfg_raw = copy.deepcopy(cfg)
    cfg_raw.optim.signed, cfg_raw.optim.grad_clip, cfg_raw.optim.langevin_noise = None, None, 0.0
    att_raw = ref.attacks.prepare_attack(model, loss_fn, cfg_raw, setup)
    att_raw.dm, att_raw.ds, att_raw.data_shape = attacker.dm, attacker.ds, attacker.data_shape
    att_raw.objective.initialize(att_raw.loss_fn, att_raw.cfg.impl, None)
    c0 = att_raw._initialize_data([n, *attacker.data_shape]); c0.data = x0.clone()
    lab0 = att_raw._initialize_data(label_template.shape); lab0.data = l0.clone()
    opt_raw, _ = att_raw._init_optimizer([c0, lab0])
    obj0 = att_raw._compute_objective(c0, lab0, rec_models, opt_raw, shared_ref, 0)()
    score = float(attacker._score_trial(best, label_template.argmax(dim=-1), rec_models, shared_ref))
    checksum = float(sum(p.double().sum() for p in model.parameters()))
    return dict(case=case_kwargs, attack=attack, overrides=overrides, iters=iters, x0=x0, l0=l0, label_template=label_template.detach().clone(),
                objective0=float(obj0), raw_grad_x0=c0.grad.detach().clone(), raw_grad_l0=lab0.grad.detach().clone(),
                task_loss0=float(att_raw.current_task_loss), history=history, lrs=lrs, candidate_final=cand.detach().clone(),
                labels_final=labels.detach().clone(), best=best, best_labels=best_l, score=score, scoring=cfg.restarts.scoring,
                true_labels=true["labels"], weight_checksum=checksum, torch_version=torch.__version__)


def config5_fixture(ref):
    """BASELINE config 5 at full size (TransformerModel(50257, 96, 8, 1536, 3), 1 x 32 tokens, tag.yaml) through the reference's
    joint attacker.  The label tensors are 1 x 32 x 50257 floats each, so the fixture keeps the candidate, the seeds from which
    the label logits are regenerated, the objective / task loss, the candidate gradient, and a strided sample + norms of the
    label-logit gradient."""
    from torch.nn.attention import SDPBackend, sdpa_kernel

    case = dict(batch=1, seq_len=32, seed=233, ntokens=50257, ninp=96, nhead=8, nhid=1536, nlayers=3)
    with sdpa_kernel(SDPBackend.MATH):
        fx = run_reference_joint(ref, case, "tag", {}, 3)
    l0, gl = fx["l0"], fx["raw_grad_l0"]
    keep = dict(case=case, attack="tag", overrides={}, iters=3, x0=fx["x0"], l0_seed=case["seed"] + 1000,
                l0_checksum=float(l0.double().sum()), l0_abs_checksum=float(l0.double().abs().sum()),
                objective0=fx["objective0"], task_loss0=fx["task_loss0"], raw_grad_x0=fx["raw_grad_x0"],
                raw_grad_l0_sample=gl[:, :, ::97].clone(), raw_grad_l0_norm=float(gl.double().norm()),
                history=fx["history"], lrs=fx["lrs"], weight_checksum=fx["weight_checksum"], torch_version=fx["torch_version"])
    return keep


def label_fixtures(ref):
    from breaching.attacks.base_attack import _BaseAttacker

    out = []
    gen = torch.Generator().manual_seed(99)
    for strategy in ["iDLG", "analytic", "yin", "wainakh-simple", "bias-corrected"]:
        for num_classes, n, repeated in [(10, 1, False), (10, 4, False), (10, 4, True), (397, 8, False), (50, 6, True)]:
            if repeated:
                y = torch.randint(0, max(2, num_classes // 4), (n,), generator=gen)
            else:
                y = torch.randperm(num_classes, generator=gen)[:n]
            feats = torch.rand(n, 16, generator=gen) + 0.1  # post-ReLU features are positive
            W = torch.randn(num_classes, 16, generator=gen, requires_grad=True)
            b = torch.zeros(num_classes, requires_grad=True)
            loss = torch.nn.functional.cross_entropy(feats @ W.t() + b, y)
            gW, gb = torch.autograd.grad(loss, (W, b))
            shared = [dict(gradients=[gW.clone(), gb.clone()], buffers=None,
                           metadata=dict(num_data_points=n, labels=None, local_hyperparams=None))]
            cfg = refshim.load_reference_attack_cfg("invertinggradients", {"label_strategy": strategy})
            att = _BaseAttacker.__new__(_BaseAttacker)
            att.cfg = cfg
            att.setup = dict(device=torch.device("cpu"), dtype=torch.float)
            torch.manual_seed(1234)  # padding with random labels draws from the global generator
            labels = att._recover_label_information(copy.deepcopy(shared), None, None)
            out.append(dict(strategy=strategy, num_classes=num_classes, n=n, gW=gW, gb=gb, true=y.sort()[0], recovered=labels))
    return out


INIT_TYPES = ["randn", "randn-trunc", "rand", "zeros", "red", "green-true", "blue", "dark", "light-true", "patterned-4", "rand-patterned-8",
              "randn-patterned-3", "wei-4", "rand-wei-5"]


def init_fixtures(ref):
    """Candidate initialisations of the reference (`_BaseAttacker._initialize_data`, base_attack.py:222-285) from a seeded global
    generator, for every scheme incl. the `patterned-k` / `wei-k` tiles and the colour fills."""
    from breaching.attacks.base_attack import _BaseAttacker

    out = []
    dm = torch.tensor(synthetic.IMAGENET["mean"])[None, :, None, None]
    ds = torch.tensor(synthetic.IMAGENET["std"])[None, :, None, None]
    for init in INIT_TYPES:
        att = _BaseAttacker.__new__(_BaseAttacker)
        att.cfg = refshim.load_reference_attack_cfg("invertinggradients", {"init": init})
        att.setup = dict(device=torch.device("cpu"), dtype=torch.float)
        att.dm, att.ds = dm, ds
        att.memory_format = torch.contiguous_format
        torch.manual_seed(4321)
        cand = att._initialize_data([2, 3, 19, 21])
        out.append(dict(init=init, shape=[2, 3, 19, 21], seed=4321, candidate=cand.detach().clone()))
    return out


def lr_fixtures(ref):
    from breaching.attacks.auxiliaries.common import optimizer_lookup
    from oracle.restate import lr_table_by_stepping

    out = []
    for sched in ["step-lr", "cosine-decay", "linear", None]:
        for warm in [0, 50]:
            for T in [300, 1000]:
                out.append(dict(scheduler=sched, warmup=warm, T=T, step_size=0.1,
                                table=lr_table_by_stepping(0.1, sched, warm, T, T, optimizer_lookup)))
    out.append(dict(scheduler="step-lr", warmup=0, T=24000, step_size=0.1,
                    table=lr_table_by_stepping(0.1, "step-lr", 0, 24000, 24000, optimizer_lookup)))
    return out


def config_fixtures():
    names = ["invertinggradients", "modern", "seethroughgradients", "clsattack", "legacy", "sanitycheck", "tag",
             "deepleakage", "beyondinfering", "wei", "multiscale_ghiasi", "_default_optimization_attack"]

    def plain(node):
        if isinstance(node, dict):
            return {k: plain(v) for k, v in node.items()}
        return node

    return {n: plain(refshim.load_reference_attack_cfg(n)) for n in names}


def dropin_fixture(ref):
    """What the drop-in tests compare against: the reference attacker's text prologue / token recovery on the miniature causal-LM
    case, and the reference's own ``TransformerModel`` (weights, autograd loss and gradients, and the layer program
    ``compile_transformer`` lowers it to).  The inputs are stored next to the outputs, so the comparison does not depend on how
    a machine's CPU kernels round."""
    import dataclasses

    from torch.nn.attention import SDPBackend, sdpa_kernel

    from breaching.cases.models.language_models import TransformerModel

    from breaching_b200 import compiler

    case = dict(batch=2, seq_len=6, seed=77)
    model, loss_fn, payload, shared, true = synthetic.make_text_case(**case)
    cfg = refshim.load_reference_attack_cfg("tag", {})
    att = ref.attacks.prepare_attack(model, loss_fn, cfg, dict(device=torch.device("cpu"), dtype=torch.float))
    shared_in = [g.clone() for g in shared[0]["gradients"]]
    sh_ref = copy.deepcopy(shared)
    rec_models, _, _ = att.prepare_attack(payload, sh_ref)
    dim = att.embeddings[0]["weight"].shape[1]
    gen = torch.Generator().manual_seed(5)
    rec_data = model.encoder.weight.detach()[true["data"]] + 0.01 * torch.randn(2, 6, dim, generator=gen)
    recovered = {}
    for mode in ("from-embedding", "from-labels", "from-limited-embedding"):
        att.cfg.token_recovery = mode
        recovered[mode] = att._postprocess_text_data(dict(data=rec_data.clone(), labels=true["data"].clone()))["data"]
    text = dict(case=case, weight_checksum=float(sum(p.double().sum() for p in model.parameters())), text_strategy=cfg.text_strategy,
                shared_gradients=shared_in, gradients_after=[g.clone() for g in sh_ref[0]["gradients"]],
                embedding_weight=att.embeddings[0]["weight"].detach().clone(), embedding_grads=att.embeddings[0]["grads"].clone(),
                dim=dim, data_shape=list(att.data_shape), param_names=[n for n, _ in rec_models[0].named_parameters()],
                encoder_is_identity=isinstance(rec_models[0].encoder, torch.nn.Identity), rec_data=rec_data, tokens=true["data"].clone(),
                recovered=recovered)

    torch.manual_seed(4)
    tm = TransformerModel(ntokens=40, ninp=16, nhead=4, nhid=24, nlayers=2, dropout=0.0, positional_embedding="learnable").eval()
    weights = [p.detach().clone() for p in tm.parameters()]        # float32: .double() below converts them exactly
    names = [n for n, _ in tm.named_parameters()]
    tm = tm.double()
    B, T = 2, 6
    program = dataclasses.asdict(compiler.compile_transformer(tm, B, T, pad_vocab=False))
    x = torch.randn(B, T, 16, dtype=torch.double, requires_grad=True)
    q = torch.softmax(torch.randn(B, T, 40, dtype=torch.double), dim=-1)
    tm.encoder = torch.nn.Identity()
    with sdpa_kernel(SDPBackend.MATH):
        loss = synthetic.causal_loss(tm(x), q)
        grads = torch.autograd.grad(loss, list(tm.parameters()))
    grads = [g.detach() for g in grads]
    # a sequence of T positions reads the first T rows of the positional table: the other rows do not enter the loss and their
    # gradient rows are exactly zero, so only the first T rows are kept
    pos = names.index("pos_encoder.embedding.weight")
    gpos = [n for n in names if n != "encoder.weight"].index("pos_encoder.embedding.weight")   # grads skip the token embedding
    assert grads[gpos][T:].abs().max().item() == 0.0
    weights[pos], grads[gpos] = weights[pos][:T].clone(), grads[gpos][:T].clone()
    transformer = dict(ctor=dict(ntokens=40, ninp=16, nhead=4, nhid=24, nlayers=2), batch=B, seq_len=T, param_names=names, weights=weights,
                       program=program, x=x.detach(), q=q, loss=float(loss), grads=grads)
    return dict(text=text, transformer=transformer, torch_version=torch.__version__)


def main():
    sys.path.insert(0, os.path.dirname(HERE))
    from helpers import FIXTURE_THREADS

    torch.set_num_threads(FIXTURE_THREADS)   # the CPU replays in tests/ run with the same count
    ref = refshim.import_reference()
    torch.manual_seed(0)
    only = sys.argv[1:]   # optional: regenerate just the named fixtures
    for name, (case_kwargs, attack, overrides, iters) in {**CASES, **FEDAVG_CASES, **LBFGS_CASES, **MULTI_QUERY_CASES, **TRAIN_BN_CASES}.items():
        if only and name not in only:
            continue
        fx = run_reference(ref, case_kwargs, attack, overrides, iters)
        torch.save(fx, os.path.join(HERE, f"trial_{name}.pt"))
        print(name, "history", [round(h, 5) for h in fx["history"]], "score", fx["score"])
    for name, (case_kwargs, attack, overrides, iters) in JOINT_CASES.items():
        if only and name not in only:
            continue
        torch.manual_seed(0)
        from torch.nn.attention import SDPBackend, sdpa_kernel

        with sdpa_kernel(SDPBackend.MATH):  # torch >= 2 fused CPU attention has no double backward (SURVEY section 8c shim 3)
            fx = run_reference_joint(ref, case_kwargs, attack, overrides, iters)
        torch.save(fx, os.path.join(HERE, f"trial_{name}.pt"))
        print(name, "history", [round(h, 5) for h in fx["history"]], "score", fx["score"])
    if not only or "joint_tag_config5" in only:
        fx = config5_fixture(ref)
        torch.save(fx, os.path.join(HERE, "trial_joint_tag_config5.pt"))
        print("joint_tag_config5 history", [round(h, 5) for h in fx["history"]])
    if "configs" in only:
        torch.save(config_fixtures(), os.path.join(HERE, "attack_configs.pt"))
    if not only or "inits" in only:
        torch.save(init_fixtures(ref), os.path.join(HERE, "inits.pt"))
    if not only or "dropin" in only:
        torch.save(dropin_fixture(ref), os.path.join(HERE, "dropin.pt"))
    if only:
        return
    torch.save(label_fixtures(ref), os.path.join(HERE, "labels.pt"))
    torch.save(lr_fixtures(ref), os.path.join(HERE, "lr_tables.pt"))
    torch.save(config_fixtures(), os.path.join(HERE, "attack_configs.pt"))
    print("fixtures written to", HERE)


if __name__ == "__main__":
    main()
