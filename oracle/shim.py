"""TEST INFRASTRUCTURE ONLY -- import shim for the *unmodified* reference.

The reference is not part of this repository: point `SWIN_REFERENCE_ROOT` at a checkout of it
(the directory holding `networks/` and `utils/`) to use it.  Its hot-path file
(`networks/swinv2_global.py:5,12`) hard-imports `ruamel.yaml` and `timm.layers`, which need not
be installed.  This module registers minimal stand-ins in `sys.modules` so the reference file can be
imported *unmodified*, where it is used for exactly two things:

  * validating `oracle/swinv2_oracle.py` (our CPU restatement) against the real reference, and
  * generating the golden fixtures under `tests/golden/` (`oracle/make_golden.py`).

Without `SWIN_REFERENCE_ROOT` the reference is absent, so nothing in `-m gpu` tests, `smoke()` or
`bench.py` may call `import_reference()`.  The product package never imports this file.

Third-party semantics restated here (timm is un-pinned by the reference; header says "Adapted from
timm v0.9.2", `swinv2_global.py:15-16`):
  * `timm.layers.Mlp`      : drop2(fc2(norm(drop1(act(fc1(x)))))), act=nn.GELU (exact erf), bias=True,
                             sub-module names fc1/act/drop1/norm/fc2/drop2 (call sites `:240-246`, `:381-386`)
  * `timm.layers.DropPath` : identity if p==0 or eval, else x * bernoulli(keep)/keep with mask (B,1,..)
                             (call sites `:378,388`)
  * `to_2tuple`, `_assert` : helpers (`:362-363,542-543`)
"""
import collections.abc
import os
import sys
import types

import torch
import torch.nn as nn

REFERENCE_ROOT = os.environ.get("SWIN_REFERENCE_ROOT", "")


def _to_2tuple(x):
    if isinstance(x, collections.abc.Iterable) and not isinstance(x, str):
        return tuple(x)
    return (x, x)


def _assert(cond, msg=""):
    assert cond, msg


class _DropPath(nn.Module):
    def __init__(self, drop_prob: float = 0.0, scale_by_keep: bool = True):
        super().__init__()
        self.drop_prob = drop_prob
        self.scale_by_keep = scale_by_keep

    def forward(self, x):
        if self.drop_prob == 0.0 or not self.training:
            return x
        keep = 1.0 - self.drop_prob
        mask = x.new_empty((x.shape[0],) + (1,) * (x.ndim - 1)).bernoulli_(keep)
        if keep > 0.0 and self.scale_by_keep:
            mask.div_(keep)
        return x * mask


class _Mlp(nn.Module):
    def __init__(self, in_features, hidden_features=None, out_features=None, act_layer=nn.GELU,
                 norm_layer=None, bias=True, drop=0.0, use_conv=False):
        super().__init__()
        out_features = out_features or in_features
        hidden_features = hidden_features or in_features
        bias = _to_2tuple(bias)
        drop = _to_2tuple(drop)
        self.fc1 = nn.Linear(in_features, hidden_features, bias=bias[0])
        self.act = act_layer()
        self.drop1 = nn.Dropout(drop[0])
        self.norm = norm_layer(hidden_features) if norm_layer is not None else nn.Identity()
        self.fc2 = nn.Linear(hidden_features, out_features, bias=bias[1])
        self.drop2 = nn.Dropout(drop[1])

    def forward(self, x):
        return self.drop2(self.fc2(self.norm(self.drop1(self.act(self.fc1(x))))))


class _ClassifierHead(nn.Module):  # imported by the reference, never used
    pass


def install():
    """Register the stand-in modules (idempotent)."""
    if "timm.layers" not in sys.modules:
        timm = types.ModuleType("timm")
        layers = types.ModuleType("timm.layers")
        layers.DropPath = _DropPath
        layers.Mlp = _Mlp
        layers.ClassifierHead = _ClassifierHead
        layers.to_2tuple = _to_2tuple
        layers._assert = _assert
        timm.layers = layers
        sys.modules["timm"] = timm
        sys.modules["timm.layers"] = layers
    if "ruamel.yaml" not in sys.modules:
        import yaml as _pyyaml

        class YAML:
            def load(self, f):
                return _pyyaml.safe_load(f)

        ruamel = types.ModuleType("ruamel")
        ryaml = types.ModuleType("ruamel.yaml")
        ryaml.YAML = YAML
        ruamel.yaml = ryaml
        sys.modules["ruamel"] = ruamel
        sys.modules["ruamel.yaml"] = ryaml
    if "torch_harmonics" not in sys.modules:
        th = types.ModuleType("torch_harmonics")
        thq = types.ModuleType("torch_harmonics.quadrature")

        def _unavailable(*a, **k):
            raise RuntimeError("torch_harmonics is not installed (only imported by the reference)")

        th.RealSHT = _unavailable
        thq.legendre_gauss_weights = _unavailable
        thq.clenshaw_curtiss_weights = _unavailable
        th.quadrature = thq
        sys.modules["torch_harmonics"] = th
        sys.modules["torch_harmonics.quadrature"] = thq


def reference_available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isfile(os.path.join(REFERENCE_ROOT, "networks", "swinv2_global.py"))


def import_reference():
    """Returns (swinv2_global module, losses module) of the unmodified reference."""
    if not reference_available():
        raise RuntimeError(f"reference tree not found: set SWIN_REFERENCE_ROOT (now {REFERENCE_ROOT!r})")
    install()
    # the reference uses top-level package names `networks` / `utils`; load them under private
    # names so they can never shadow (or be shadowed by) anything of ours
    import importlib.util

    def _load(name, rel):
        spec = importlib.util.spec_from_file_location(name, os.path.join(REFERENCE_ROOT, rel))
        mod = importlib.util.module_from_spec(spec)
        sys.modules[name] = mod
        spec.loader.exec_module(mod)
        return mod

    if "_ref_swinv2_global" in sys.modules:
        return sys.modules["_ref_swinv2_global"], sys.modules["_ref_losses"]
    swin = _load("_ref_swinv2_global", "networks/swinv2_global.py")
    # utils.losses does `from utils.grids import GridQuadrature`
    saved = {k: sys.modules.get(k) for k in ("utils", "utils.grids")}
    pkg = types.ModuleType("utils")
    pkg.__path__ = [os.path.join(REFERENCE_ROOT, "utils")]
    sys.modules["utils"] = pkg
    grids = _load("utils.grids", "utils/grids.py")
    losses = _load("_ref_losses", "utils/losses.py")
    sys.modules["_ref_grids"] = grids
    for k, v in saved.items():
        if v is None:
            sys.modules.pop(k, None)
        else:
            sys.modules[k] = v
    return swin, losses
