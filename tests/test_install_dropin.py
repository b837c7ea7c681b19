"""Drop-in mounting: ``breaching_b200.install.install()`` rebinds ``breaching.attacks.prepare_attack`` of the (unmodified)
reference package, so reference entry points keep calling ``breaching.attacks.prepare_attack(...)`` unchanged.

The rebinding is exercised on a stand-in ``breaching`` package written to a temporary directory; the comparisons with the
reference run against what the reference computed on the same inputs, stored under ``tests/golden/`` (``attack_configs.pt``,
``dropin.pt``; recipe in ``tests/golden/make_golden.py``)."""
import dataclasses
import sys

import pytest
import torch

from oracle import refshim

_STAND_IN = '''
calls = []


def prepare_attack(model, loss, cfg_attack, setup):
    calls.append(cfg_attack.attack_type)
    return ("reference attacker", cfg_attack.attack_type)
'''


@pytest.fixture
def stand_in_reference(tmp_path, monkeypatch):
    """A minimal importable ``breaching`` package whose ``attacks.prepare_attack`` records its calls."""
    from breaching_b200 import install as inst

    pkg = tmp_path / "breaching"
    (pkg / "attacks").mkdir(parents=True)
    (pkg / "__init__.py").write_text("from . import attacks  # noqa: F401\n")
    (pkg / "attacks" / "__init__.py").write_text(_STAND_IN)
    for name in [m for m in sys.modules if m == "breaching" or m.startswith("breaching.")]:
        monkeypatch.delitem(sys.modules, name)
    monkeypatch.syspath_prepend(str(tmp_path))
    monkeypatch.setattr(inst, "_ORIGINAL", None)
    import breaching

    assert breaching.__file__.startswith(str(tmp_path))
    return breaching


def test_install_rebinds_prepare_attack_and_delegates_other_attack_types(stand_in_reference):
    ref = stand_in_reference
    import breaching_b200
    from breaching_b200 import install as inst
    from breaching_b200 import synthetic
    from breaching_b200.engine import EngineError

    original = ref.attacks.prepare_attack
    try:
        returned = inst.install()
        assert returned is original
        assert ref.attacks.prepare_attack.__module__.startswith("breaching_b200")
        model = synthetic.build_model("convnet-tiny", 10)
        loss = torch.nn.CrossEntropyLoss()
        setup = dict(device=torch.device("cpu"), dtype=torch.float)
        # optimisation attacks go to the B200 engine: on a CPU "device" it refuses loudly (no fallback) ...
        with pytest.raises(EngineError):
            ref.attacks.prepare_attack(model, loss, breaching_b200.get_attack_config("invertinggradients"), setup)
        assert ref.attacks.calls == []
        # ... while the attack types outside the accelerated path are delegated to the reference's own prepare_attack
        cfg = refshim.RefCfg(attack_type="analytic")
        assert ref.attacks.prepare_attack(model, loss, cfg, setup) == ("reference attacker", "analytic")
        assert ref.attacks.calls == ["analytic"]
    finally:
        inst.uninstall()
    assert ref.attacks.prepare_attack is original


def test_reference_yaml_config_objects_are_accepted_by_the_engine_config_flattening(golden):
    """cfg objects composed from the reference's own YAML (attribute + item access) flatten to the same C struct as ours."""
    import ctypes

    import breaching_b200
    from breaching_b200.engine import make_cfg

    ref_cfgs = golden("attack_configs.pt")
    for name in ["invertinggradients", "modern", "seethroughgradients", "clsattack", "legacy"]:
        a = make_cfg(refshim._coerce(ref_cfgs[name]))
        b = make_cfg(breaching_b200.get_attack_config(name))
        assert bytes(ctypes.string_at(ctypes.addressof(a), ctypes.sizeof(a))) == bytes(ctypes.string_at(ctypes.addressof(b), ctypes.sizeof(b))), name


def test_text_prologue_and_token_recovery_match_the_reference(golden):
    """host.prepare_for_text_data / postprocess_text_data against the reference attacker's own methods
    (base_attack.py:76-167) on the miniature causal-LM case."""
    import copy

    from breaching_b200 import synthetic
    from breaching_b200.attacks import host

    fx = golden("dropin.pt")["text"]
    model, loss_fn, payload, shared, true = synthetic.make_text_case(**fx["case"])
    checksum = float(sum(p.double().sum() for p in model.parameters()))
    assert abs(checksum - fx["weight_checksum"]) <= 1e-6 * max(1.0, abs(fx["weight_checksum"])), "synthetic text case changed"
    # the shared update the reference received (CPU autograd rounding may differ between machines)
    sh_mine = copy.deepcopy(shared)
    sh_mine[0]["gradients"] = [g.clone() for g in fx["shared_gradients"]]
    mine = copy.deepcopy(model)
    emb, dim = host.prepare_for_text_data([mine], sh_mine, fx["text_strategy"])
    assert dim == fx["dim"] == fx["data_shape"][-1]
    assert len(sh_mine[0]["gradients"]) == len(fx["gradients_after"])
    for a, b in zip(sh_mine[0]["gradients"], fx["gradients_after"]):
        assert torch.equal(a, b)
    assert torch.equal(emb[0]["grads"], fx["embedding_grads"])
    assert torch.equal(emb[0]["weight"].detach(), fx["embedding_weight"])
    assert isinstance(mine.encoder, torch.nn.Identity) and fx["encoder_is_identity"]
    assert [n for n, _ in mine.named_parameters()] == fx["param_names"]
    # token recovery from reconstructed embeddings: noisy true embeddings must map back to the tokens, identically to the reference
    for mode, expect in fx["recovered"].items():
        got = host.postprocess_text_data(dict(data=fx["rec_data"].clone(), labels=fx["tokens"].clone()), emb[0]["weight"].detach(), mode)
        assert torch.equal(got["data"], expect), mode


def test_compile_transformer_accepts_the_reference_model_class(golden):
    """``compiler.compile_transformer`` and the reference's own ``TransformerModel`` (cases/models/language_models.py:150-205):
    ``synthetic.TransformerLM`` with the reference instance's weights has the same parameter names and order and lowers to the
    program the reference instance lowered to; that program, run by the four-sweep interpreter, reproduces the loss and
    gradients autograd computed through the reference module."""
    from breaching_b200 import compiler, synthetic
    from oracle import program_interp as PI

    fx = golden("dropin.pt")["transformer"]
    B, T = fx["batch"], fx["seq_len"]
    mine = synthetic.TransformerLM(**fx["ctor"]).double()
    names = [n for n, _ in mine.named_parameters()]
    assert names == fx["param_names"]
    with torch.no_grad():
        for p, w in zip(mine.parameters(), fx["weights"]):
            p.zero_()
            p[: w.shape[0]].copy_(w)       # the positional table is stored up to the T rows a sequence reads
    prog = compiler.compile_transformer(mine, B, T, pad_vocab=False)   # the torch interpreter runs the un-padded program
    assert dataclasses.asdict(prog) == fx["program"]
    mine.encoder = torch.nn.Identity()                      # what the attack does (base_attack.py:100-110)
    params = [p for p in mine.parameters()]

    class _Params:
        def parameters(self):
            return params

        def named_modules(self):
            return mine.named_modules()

    it = PI.ProgramInterpreter(_Params(), prog)
    assert abs(float(it.forward(fx["x"], fx["q"])) - fx["loss"]) < 1e-12
    grads = it.backward()
    assert len(grads) == len(fx["grads"])
    for a, b in zip(grads, fx["grads"]):
        rows = b.shape[0]
        assert a[rows:].abs().sum().item() == 0.0                  # positional rows the sequence does not read
        assert ((a[:rows] - b).norm() / (b.norm() + 1e-300)).item() < 1e-10
