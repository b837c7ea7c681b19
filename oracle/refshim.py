"""Import the *unmodified* reference (``/root/reference/breaching``) in this container.

TEST INFRASTRUCTURE ONLY.  Works only where ``/root/reference`` exists (the build
container); the GPU box has no reference tree, so nothing on the ``-m gpu`` path,
``smoke()`` or ``bench.py`` touches this module.  It is used by
``tests/golden/make_golden.py`` to produce the committed fixtures; the tests use
only its ``RefCfg`` config objects and compare against those fixtures.

Shims (SURVEY.md section 8c):
  * ``hydra`` / ``omegaconf`` are not installed -> stub modules in ``sys.modules``
    before ``import breaching`` (reference ``breaching/__init__.py:11``,
    ``breaching/utils.py:17-18`` import them at module top).
  * the attack config is composed from the reference's own YAML files with PyYAML,
    reproducing the OmegaConf behaviours the attacker relies on: ``defaults:``
    merging, attribute + item access, ``1e-4`` parsed as float (PyYAML reads it as
    a string), ``None`` staying the *string* "None" (``tag.yaml:9``).
"""
import os
import re
import sys
import types

REFERENCE_ROOT = os.environ.get("BREACHING_REFERENCE_ROOT", "/root/reference")


def reference_available():
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "breaching"))


class RefCfg(dict):
    """Minimal OmegaConf-DictConfig look-alike: attribute access, item access, ``keys()``/``items()``."""

    def __getattr__(self, key):
        try:
            return self[key]
        except KeyError as exc:  # AttributeError so that ``hasattr``/``try: ... except AttributeError`` work
            raise AttributeError(key) from exc

    def __setattr__(self, key, value):
        self[key] = value


_FLOAT_RE = re.compile(r"^[+-]?(\d+\.?\d*|\.\d+)([eE][+-]?\d+)?$")


def _coerce(value):
    if isinstance(value, dict):
        return RefCfg({k: _coerce(v) for k, v in value.items()})
    if isinstance(value, list):
        return [_coerce(v) for v in value]
    if isinstance(value, str) and _FLOAT_RE.match(value.replace("_", "")) and any(c in value for c in ".eE"):
        return float(value.replace("_", ""))
    return value


def _merge(base, new):
    for key, val in new.items():
        if isinstance(val, dict) and isinstance(base.get(key), dict):
            _merge(base[key], val)
        else:
            base[key] = val
    return base


def load_reference_attack_cfg(name, overrides=None):
    """Compose ``breaching/config/attack/<name>.yaml`` (+ its ``defaults:``) the way hydra would."""
    import yaml

    folder = os.path.join(REFERENCE_ROOT, "breaching", "config", "attack")

    def load(fname):
        with open(os.path.join(folder, fname + ".yaml")) as handle:
            raw = yaml.safe_load(handle) or {}
        merged = {}
        for entry in raw.pop("defaults", []):
            if entry == "_self_":
                continue
            _merge(merged, load(entry))
        return _merge(merged, raw)

    cfg = _coerce(load(name))
    for dotted, value in (overrides or {}).items():
        node = cfg
        parts = dotted.split(".")
        for part in parts[:-1]:
            if node.get(part) is None:
                node[part] = RefCfg()
            node = node[part]
        node[parts[-1]] = _coerce(value)
    return cfg


def import_reference():
    """Return the reference's ``breaching`` package (stubbing hydra/omegaconf)."""
    if not reference_available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    if "breaching" in sys.modules and getattr(sys.modules["breaching"], "__file__", "").startswith(REFERENCE_ROOT):
        return sys.modules["breaching"]
    for modname in ["hydra", "hydra.utils", "hydra.core", "hydra.core.hydra_config", "omegaconf"]:
        if modname not in sys.modules:
            stub = types.ModuleType(modname)
            stub.__path__ = []
            sys.modules[modname] = stub
    sys.modules["omegaconf"].OmegaConf = type("OmegaConf", (), {"to_yaml": staticmethod(lambda cfg: str(cfg))})
    sys.modules["omegaconf"].open_dict = lambda cfg: cfg
    sys.modules["hydra"].utils = sys.modules["hydra.utils"]
    sys.modules["hydra.utils"].get_original_cwd = os.getcwd
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import breaching  # noqa: E402  (the reference)

    return breaching
