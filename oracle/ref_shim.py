"""Import the UNMODIFIED reference (a checkout of CGCL-codes/DorPatch) on a CPU-only box.

Used only by ``tests/golden/make_golden.py`` to generate the golden vectors the
test suite pins the oracle against; the suite itself never needs the reference.
Nothing is copied: the reference modules are imported from where they lie.

Shim (SURVEY.md section 8c):
  * ``Tensor.cuda`` / ``Tensor.cpu`` return a *copy* on the CPU (on a GPU box
    both are device transfers that never alias their source; an identity shim
    would make the reference's ``adv_pattern_best_np = adv_x.cpu().numpy()``
    (attack.py:159) alias the live pattern and silently change its result);
    ``Module.cuda`` is identity;
  * ``timm`` (not installed, third-party) is replaced by an empty stub module --
    ``utils.get_model`` is never called, the caller passes its own model;
  * the reference checkout is put on ``sys.path`` so ``attack``, ``utils`` and
    ``defenses.PatchCleanser`` resolve to the reference's files.
TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).
"""
import contextlib
import importlib
import importlib.util
import os
import sys
import types

_REF_MODULES = ("attack", "utils", "defenses", "defenses.PatchCleanser", "main")


def available(root):
    return os.path.isfile(os.path.join(root, "attack.py"))


@contextlib.contextmanager
def reference_modules(root):
    """Context manager yielding a namespace with the reference's ``attack``,
    ``utils`` and ``PatchCleanser`` modules; restores sys.modules/sys.path and
    the torch monkeypatches on exit so the product's same-named root modules
    are unaffected."""
    import torch
    import torchvision  # noqa: F401  (the reference imports it)
    saved = {k: sys.modules.get(k) for k in _REF_MODULES + ("timm",)}
    saved_path = list(sys.path)
    t_cuda, t_cpu, m_cuda = torch.Tensor.cuda, torch.Tensor.cpu, torch.nn.Module.cuda
    try:
        for k in _REF_MODULES:
            sys.modules.pop(k, None)
        sys.modules["timm"] = types.ModuleType("timm")
        sys.path.insert(0, root)
        torch.Tensor.cuda = lambda self, *a, **k: self.clone()
        torch.Tensor.cpu = lambda self, *a, **k: self.clone()
        torch.nn.Module.cuda = lambda self, *a, **k: self
        ns = types.SimpleNamespace()
        # Load by file path: the repo root holds same-named drop-in modules (attack, utils,
        # defenses/ -- a regular package, which would shadow the reference's namespace package).
        pkg = types.ModuleType("defenses")
        pkg.__path__ = [os.path.join(root, "defenses")]
        sys.modules["defenses"] = pkg

        def load(name, rel):
            spec = importlib.util.spec_from_file_location(name, os.path.join(root, rel))
            mod = importlib.util.module_from_spec(spec)
            sys.modules[name] = mod
            spec.loader.exec_module(mod)
            return mod

        ns.utils = load("utils", "utils.py")
        ns.PatchCleanser = load("defenses.PatchCleanser", "defenses/PatchCleanser.py")
        ns.attack = load("attack", "attack.py")
        assert ns.attack.__file__.startswith(root), ns.attack.__file__
        assert ns.attack.MaskWindow is ns.PatchCleanser.MaskWindow and ns.attack.clip is ns.utils.clip
        yield ns
    finally:
        torch.Tensor.cuda, torch.Tensor.cpu, torch.nn.Module.cuda = t_cuda, t_cpu, m_cuda
        sys.path[:] = saved_path
        for k in _REF_MODULES + ("timm",):
            sys.modules.pop(k, None)
            if saved[k] is not None:
                sys.modules[k] = saved[k]
