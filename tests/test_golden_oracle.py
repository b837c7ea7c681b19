"""Pin the CPU oracle (oracle/restate.py) against the fixtures produced by the unmodified reference."""
import math

import pytest
import torch

from helpers import (FEDAVG_FIXTURES, JOINT_FIXTURES, LBFGS_FIXTURES, MULTI_QUERY_FIXTURES, TRAIN_BN_FIXTURES, TRIAL_FIXTURES,
                     fixture_threads, joint_oracle_for_fixture,
                     load_golden, multi_query_oracle_for_fixture, oracle_for_fixture)


@pytest.fixture(autouse=True)
def _same_threads_as_the_fixtures():
    with fixture_threads():
        yield


@pytest.mark.parametrize("name", TRIAL_FIXTURES + FEDAVG_FIXTURES + LBFGS_FIXTURES + TRAIN_BN_FIXTURES)
def test_oracle_reproduces_reference_trajectory(name):
    fx = load_golden(f"trial_{name}.pt")
    orc, cfg, labels = oracle_for_fixture(fx)
    assert labels.tolist() == fx["labels"].tolist()  # label recovery: bit-exact
    phi0, _, raw, terms = orc.closure_gradient(fx["x0"], 0, 0.0)
    assert math.isclose(float(phi0), fx["objective0"], rel_tol=1e-5, abs_tol=1e-7)
    rel = ((raw - fx["raw_grad0"]).norm() / fx["raw_grad0"].norm()).item()
    assert rel < 1e-4, rel
    best, hist, trace = orc.run(fx["x0"], iterations=fx["iters"], record=True)
    assert len(hist) == len(fx["history"])
    # L-BFGS takes 20 inner iterations per recorded value: float32 summation-order differences (and, with the default hard
    # sign, flipped entries of near-zero gradients) are amplified by the curvature estimate
    tol = 3e-2 if name in LBFGS_FIXTURES else 2e-4
    for a, b in zip(hist, fx["history"]):
        assert math.isclose(a, b, rel_tol=tol, abs_tol=1e-6), (hist, fx["history"])
    for t, lr in zip(trace, fx["lrs"]):
        assert math.isclose(t["lr"], lr, rel_tol=1e-9, abs_tol=1e-12)
    assert (trace[0]["candidate"] - fx["candidate_after_1"]).abs().max().item() < (5e-2 if name in LBFGS_FIXTURES else 1e-4)
    # later iterates may differ where a hard sign flips on a near-zero gradient entry: compare in the mean
    assert (trace[-1]["candidate"] - fx["candidate_final"]).abs().mean().item() < (2e-2 if name in LBFGS_FIXTURES else 2e-3)
    score = orc.score(best, fx["scoring"])
    assert math.isclose(score, fx["score"], rel_tol=5e-2, abs_tol=1e-5)
    orc.close()


@pytest.mark.parametrize("name", JOINT_FIXTURES)
def test_joint_oracle_reproduces_reference_trajectory(name):
    """attack_type joint-optimization (optimization_with_label_attack.py): soft labels optimised with the data."""
    fx = load_golden(f"trial_{name}.pt")
    orc, cfg = joint_oracle_for_fixture(fx)
    cfg_raw = dict(cfg["optim"])
    phi0, _, _, raw, terms = orc.closure_gradients(fx["x0"], fx["l0"], 0, 0.0)
    assert math.isclose(float(phi0), fx["objective0"], rel_tol=1e-5, abs_tol=1e-7)
    assert ((raw[0] - fx["raw_grad_x0"]).norm() / fx["raw_grad_x0"].norm()).item() < 1e-4
    assert ((raw[1] - fx["raw_grad_l0"]).norm() / fx["raw_grad_l0"].norm()).item() < 1e-4
    best, best_l, hist, x_final, l_final = orc.run_joint(fx["x0"], fx["l0"], iterations=fx["iters"])
    tol = 3e-2 if cfg_raw["optimizer"].lower() == "l-bfgs" else 2e-4
    assert len(hist) == len(fx["history"])
    for a, b in zip(hist, fx["history"]):
        assert math.isclose(a, b, rel_tol=tol, abs_tol=1e-5), (hist, fx["history"])
    assert (x_final - fx["candidate_final"]).abs().mean().item() < (2e-2 if tol > 1e-3 else 2e-3)
    assert (l_final - fx["labels_final"]).abs().mean().item() < (2e-2 if tol > 1e-3 else 2e-3)
    orc.close()


@pytest.mark.parametrize("name", MULTI_QUERY_FIXTURES)
def test_multi_query_oracle_reproduces_reference_trajectory(name):
    """Two model queries on the same user batch (optimization_based_attack.py:157-160)."""
    fx = load_golden(f"trial_{name}.pt")
    orc, cfg, labels = multi_query_oracle_for_fixture(fx)
    assert labels.tolist() == fx["labels"].tolist()
    phi0, _, raw, _ = orc.closure_gradient(fx["x0"], 0, 0.0)
    assert math.isclose(float(phi0), fx["objective0"], rel_tol=1e-5, abs_tol=1e-7)
    assert ((raw - fx["raw_grad0"]).norm() / fx["raw_grad0"].norm()).item() < 1e-4
    best, hist, _ = orc.run(fx["x0"], iterations=fx["iters"])
    for a, b in zip(hist, fx["history"]):
        assert math.isclose(a, b, rel_tol=2e-4, abs_tol=1e-6), (hist, fx["history"])
    assert math.isclose(orc.score(best, fx["scoring"]), fx["score"], rel_tol=5e-2, abs_tol=1e-5)
    orc.close()


def test_lr_tables_match_reference_schedulers():
    from breaching_b200.schedule import lr_table
    from oracle import restate

    for fx in load_golden("lr_tables.pt"):
        for fn in (lr_table, restate.lr_table):
            table = fn(fx["step_size"], fx["scheduler"], fx["warmup"], fx["T"])
            assert len(table) == len(fx["table"])
            worst = max(abs(a - b) for a, b in zip(table, fx["table"]))
            assert worst < 1e-12, (fx["scheduler"], fx["warmup"], fx["T"], worst)


def test_label_recovery_bit_exact():
    from breaching_b200.attacks import host
    from oracle import restate

    setup = dict(device=torch.device("cpu"), dtype=torch.float)
    for fx in load_golden("labels.pt"):
        shared = [dict(gradients=[fx["gW"].clone(), fx["gb"].clone()], buffers=None,
                       metadata=dict(num_data_points=fx["n"], labels=None, local_hyperparams=None))]
        torch.manual_seed(1234)
        ours = host.recover_labels(fx["strategy"], shared, setup)
        assert ours.tolist() == fx["recovered"].tolist(), fx["strategy"]
        shared = [dict(gradients=[fx["gW"].clone(), fx["gb"].clone()], buffers=None,
                       metadata=dict(num_data_points=fx["n"], labels=None, local_hyperparams=None))]
        torch.manual_seed(1234)
        orc = restate.recover_labels(fx["strategy"], shared, fx["n"])
        assert orc.tolist() == fx["recovered"].tolist(), fx["strategy"]


def test_candidate_initialisation_equals_the_reference():
    """Every initialisation scheme (base_attack.py:222-285, incl. `patterned-k` / `wei-k` tiles and colour fills) from the same
    seeded generator: the product's host code and the oracle draw exactly what the reference drew."""
    from breaching_b200 import synthetic
    from breaching_b200.attacks import host
    from oracle import restate

    setup = dict(device=torch.device("cpu"), dtype=torch.float)
    dm = torch.tensor(synthetic.IMAGENET["mean"])[None, :, None, None]
    ds = torch.tensor(synthetic.IMAGENET["std"])[None, :, None, None]
    fixtures = load_golden("inits.pt")
    assert len(fixtures) >= 14
    for fx in fixtures:
        torch.manual_seed(fx["seed"])
        ours = host.initialize_data(fx["init"], fx["shape"], dm, ds, setup)
        assert torch.equal(ours, fx["candidate"]), fx["init"]
        torch.manual_seed(fx["seed"])
        orc = restate.initialize_data(fx["init"], fx["shape"], dm, ds)
        assert torch.equal(orc, fx["candidate"]), fx["init"]
    with pytest.raises(ValueError):
        host.initialize_data("no-such-scheme", [1, 3, 4, 4], dm, ds, setup)


def test_attack_presets_equal_reference_yaml():
    from breaching_b200 import config as bcfg

    def plain(node):
        return {k: plain(v) for k, v in node.items()} if isinstance(node, dict) else node

    for name, ref_cfg in load_golden("attack_configs.pt").items():
        ours = plain(bcfg.get_attack_config(name))
        assert ours == ref_cfg, name
