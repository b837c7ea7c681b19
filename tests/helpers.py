"""Shared helpers for the parity tests."""
import contextlib
import copy
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from breaching_b200 import config as bcfg  # noqa: E402
from breaching_b200 import synthetic  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")

# The trajectory fixtures were generated with 8 intra-op CPU threads (tests/golden/make_golden.py).  CPU kernels split their
# reductions by the thread count, and the FedAvg, train-mode BN and L-BFGS / joint trajectories amplify the resulting last-bit
# differences past the tolerances of the CPU replays (FedAvg's first objective moves by 2e-4 relative below 8 threads), so
# those replays run with the same count on any host.
FIXTURE_THREADS = 8


@contextlib.contextmanager
def fixture_threads():
    old = torch.get_num_threads()
    torch.set_num_threads(FIXTURE_THREADS)
    try:
        yield
    finally:
        torch.set_num_threads(old)


class OddChannelNet(torch.nn.Module):
    """3 -> 6 -> 10 -> 14 channels (none a multiple of 4: the scalar element-wise kernels), a residual add onto a tensor that also
    feeds a convolution (accumulated deltas), 3/2/1 max-pooling after a ReLU on a 15 x 13 map, average pooling, 7 classes."""

    def __init__(self, classes=7):
        super().__init__()
        nn = torch.nn
        self.conv0, self.bn0 = nn.Conv2d(3, 6, 3, padding=1), nn.BatchNorm2d(6)
        self.conv1, self.bn1 = nn.Conv2d(6, 10, 3, padding=1, bias=False), nn.BatchNorm2d(10)
        self.conv2, self.bn2 = nn.Conv2d(10, 10, 3, padding=1, bias=False), nn.BatchNorm2d(10)
        self.pool = nn.MaxPool2d(3, 2, 1)
        self.conv3, self.bn3 = nn.Conv2d(10, 14, 3, padding=1), nn.BatchNorm2d(14)
        self.avg = nn.AdaptiveAvgPool2d(1)
        self.fc = nn.Linear(14, classes)

    def forward(self, x):
        h = torch.relu(self.bn0(self.conv0(x)))
        h1 = torch.relu(self.bn1(self.conv1(h)))
        h2 = torch.relu(self.bn2(self.conv2(h1)) + h1)
        h3 = torch.relu(self.bn3(self.conv3(self.pool(h2))))
        return self.fc(torch.flatten(self.avg(h3), 1))


class TensorCoreNet(torch.nn.Module):
    """Channel counts the tcgen05 kernels take with both tile widths: a 3-channel stem, 32 -> 96 and 96 -> 64 layers (128 x 32
    tiles), 64-channel layers (128 x 64 tiles), a stride-2 3 x 3 convolution and a 1 x 1 stride-2 downsample added back."""

    def __init__(self, classes=10):
        super().__init__()
        nn = torch.nn
        self.stem, self.bn0 = nn.Conv2d(3, 32, 3, padding=1, bias=False), nn.BatchNorm2d(32)
        self.conv1, self.bn1 = nn.Conv2d(32, 96, 3, padding=1, bias=False), nn.BatchNorm2d(96)
        self.conv2, self.bn2 = nn.Conv2d(96, 64, 3, padding=1, bias=False), nn.BatchNorm2d(64)
        self.conv3, self.bn3 = nn.Conv2d(64, 64, 3, stride=2, padding=1, bias=False), nn.BatchNorm2d(64)
        self.conv4, self.bn4 = nn.Conv2d(64, 64, 3, padding=1, bias=False), nn.BatchNorm2d(64)
        self.down, self.bnd = nn.Conv2d(64, 64, 1, stride=2, bias=False), nn.BatchNorm2d(64)
        self.avg = nn.AdaptiveAvgPool2d(1)
        self.fc = nn.Linear(64, classes)

    def forward(self, x):
        h = torch.relu(self.bn0(self.stem(x)))
        h = torch.relu(self.bn1(self.conv1(h)))
        h = torch.relu(self.bn2(self.conv2(h)))
        y = torch.relu(self.bn3(self.conv3(h)))
        y = torch.relu(self.bn4(self.conv4(y)) + self.bnd(self.down(h)))
        return self.fc(torch.flatten(self.avg(y), 1))


def parity_model(name, seed=0, train_bn=False):
    """``odd`` / ``tensor-core``: randomly initialised, BN with random affine parameters and running statistics (eval mode), or
    train-mode BN without running statistics (``train_bn``)."""
    torch.manual_seed(seed)
    model = OddChannelNet() if name == "odd" else TensorCoreNet()
    synthetic.randomize_bn(model, seed + 1)
    model.eval()
    if train_bn:
        model.train()
        for mod in model.modules():
            if isinstance(mod, torch.nn.BatchNorm2d):
                mod.track_running_stats = False
    return model


def load_golden(name):
    return torch.load(os.path.join(GOLDEN, name), weights_only=False)


def cfg_from_fixture(fx):
    return bcfg.get_attack_config(fx["attack"], dict(fx["overrides"]))


def case_from_fixture(fx):
    if "seq_len" in fx["case"]:
        model, loss_fn, payload, shared, true = synthetic.make_text_case(**fx["case"])
    elif "steps" in fx["case"]:
        model, loss_fn, payload, shared, true = synthetic.make_fedavg_case(**fx["case"])
    elif "queries" in fx["case"]:
        model, loss_fn, payload, shared, true = synthetic.make_multi_query_case(**fx["case"])
    else:
        model, loss_fn, payload, shared, true = synthetic.make_case(**fx["case"])
    checksum = float(sum(p.double().sum() for p in model.parameters()))
    assert abs(checksum - fx["weight_checksum"]) <= 1e-6 * max(1.0, abs(fx["weight_checksum"])), \
        "synthetic case differs from the one the fixture was generated with"
    return model, loss_fn, payload, shared, true


def oracle_for_fixture(fx):
    """TrialOracle (CPU restatement) set up exactly like the reference attacker was for this fixture."""
    from oracle import restate

    model, loss_fn, payload, shared, true = case_from_fixture(fx)
    cfg = cfg_from_fixture(fx)
    shared = copy.deepcopy(shared)
    m = copy.deepcopy(model)
    if shared[0]["buffers"] is not None:
        for buf, src in zip(m.buffers(), shared[0]["buffers"]):
            buf.data.copy_(src)
    m.eval()
    if shared[0]["buffers"] is None and payload[0]["buffers"] is None:  # base_attack.py:192-197: no buffers anywhere -> train mode
        m.train()
        for mod in m.modules():
            if hasattr(mod, "track_running_stats"):
                mod.track_running_stats = False
    meta = payload[0]["metadata"]
    dm = torch.tensor(meta.mean)[None, :, None, None]
    ds = torch.tensor(meta.std)[None, :, None, None]
    labels = restate.recover_labels(cfg.label_strategy, shared, shared[0]["metadata"]["num_data_points"])
    return restate.TrialOracle(m, loss_fn, cfg, shared[0]["gradients"], labels, dm, ds,
                               local_hyperparams=shared[0]["metadata"]["local_hyperparams"]), cfg, labels


TRIAL_FIXTURES = ["ig_convnet", "ig_resnet18", "stg_resnet18", "modern_convnet", "tag_clip_convnet", "l1_sgd_convnet"]
FEDAVG_FIXTURES = ["fedavg_convnet", "fedavg_resnet18"]
LBFGS_FIXTURES = ["lbfgs_convnet", "lbfgs_wei_convnet", "lbfgs_cosine_convnet"]
JOINT_FIXTURES = ["joint_dlg_convnet", "joint_adam_convnet", "joint_tag_transformer"]
MULTI_QUERY_FIXTURES = ["multiquery_convnet"]
TRAIN_BN_FIXTURES = ["trainbn_convnet", "trainbn_resnet18"]


def joint_oracle_for_fixture(fx):
    """JointTrialOracle (CPU restatement of OptimizationJointAttacker) for a joint-optimisation fixture."""
    from oracle import restate

    model, loss_fn, payload, shared, true = case_from_fixture(fx)
    cfg = cfg_from_fixture(fx)
    m = copy.deepcopy(model).eval()
    meta = payload[0]["metadata"]
    grads = list(shared[0]["gradients"])
    if getattr(meta, "modality", "vision") == "text":
        # base_attack.py:76-128 ("run-embedding"): optimise in embedding space -- drop the token-embedding gradient and bypass
        # the embedding layer; no input normalisation
        names = [n for n, _ in m.named_parameters()]
        grads.pop(names.index("encoder.weight"))
        m.encoder = torch.nn.Identity()
        dm, ds = torch.tensor(0.0), torch.tensor(1.0)
    else:
        dm = torch.tensor(meta.mean)[None, :, None, None]
        ds = torch.tensor(meta.std)[None, :, None, None]
    return restate.JointTrialOracle(m, loss_fn, cfg, grads, None, dm, ds), cfg


def multi_query_oracle_for_fixture(fx):
    """MultiQueryOracle: one TrialOracle per (model, update) pair, regularisers only on the first."""
    from oracle import restate

    model, loss_fn, payload, shared, true = case_from_fixture(fx)
    cfg = cfg_from_fixture(fx)
    no_priors = copy.deepcopy(cfg)
    if no_priors.get("regularization") is not None:
        for key in no_priors["regularization"].keys():
            no_priors["regularization"][key]["scale"] = 0.0
    meta = payload[0]["metadata"]
    dm = torch.tensor(meta.mean)[None, :, None, None]
    ds = torch.tensor(meta.std)[None, :, None, None]
    labels = restate.recover_labels(cfg.label_strategy, copy.deepcopy(shared), shared[0]["metadata"]["num_data_points"])
    oracles = []
    for i, (pl, sh) in enumerate(zip(payload, shared)):
        m = copy.deepcopy(model)
        with torch.no_grad():
            for p, src in zip(m.parameters(), pl["parameters"]):
                p.copy_(src)
            for b, src in zip(m.buffers(), pl["buffers"]):
                b.copy_(src)
        m.eval()
        oracles.append(restate.TrialOracle(m, loss_fn, cfg if i == 0 else no_priors, sh["gradients"], labels, dm, ds))
    return restate.MultiQueryOracle(oracles), cfg, labels
