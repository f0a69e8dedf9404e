"""Import shims so the UNMODIFIED reference (/root/reference) runs on CPU in the build container.

TEST INFRASTRUCTURE ONLY.  Nothing in the product path (packnet_sfm_b200/) may import this.
It is used by oracle/gen_golden.py, which generates the fixtures under tests/golden/ where the
reference tree is present; the tests read only those fixtures.

Shims (none touches arithmetic; SURVEY.md §8c):
  * stub `yacs` / `yacs.config.CfgNode`      (packnet_sfm/utils/types.py:3,41-43 — isinstance helper only)
  * stub `matplotlib.cm.get_cmap`             (packnet_sfm/utils/depth.py:6 — visualisation only)
  * `torch.Tensor.get_device` -> `.device` for CPU tensors
        (packnet_sfm/losses/multiview_photometric_loss.py:150 calls get_device() -> -1 -> Camera.to(-1) raises)
"""
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("PACKNET_REFERENCE_ROOT", "/root/reference")


def reference_available():
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "packnet_sfm"))


def install():
    """Make `import packnet_sfm...` resolve to the unmodified reference. Idempotent."""
    if not reference_available():
        raise RuntimeError("reference tree not found at %s" % REFERENCE_ROOT)
    import torch

    if "yacs" not in sys.modules:
        yacs = types.ModuleType("yacs")
        yacs_config = types.ModuleType("yacs.config")

        class CfgNode(dict):
            pass

        yacs_config.CfgNode = CfgNode
        yacs.config = yacs_config
        sys.modules["yacs"] = yacs
        sys.modules["yacs.config"] = yacs_config
    try:
        import matplotlib.cm  # noqa: F401
    except Exception:
        mpl = types.ModuleType("matplotlib")
        cm = types.ModuleType("matplotlib.cm")
        cm.get_cmap = lambda *a, **k: None
        mpl.cm = cm
        sys.modules["matplotlib"] = mpl
        sys.modules["matplotlib.cm"] = cm

    if "termcolor" not in sys.modules:
        try:
            import termcolor  # noqa: F401
        except Exception:
            tc = types.ModuleType("termcolor")
            tc.colored = lambda text, *a, **k: text
            sys.modules["termcolor"] = tc

    if not getattr(torch.Tensor.get_device, "_pn_shim", False):
        _orig = torch.Tensor.get_device

        def get_device(self):
            return _orig(self) if self.is_cuda else self.device

        get_device._pn_shim = True
        torch.Tensor.get_device = get_device

    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    # a previously installed drop-in must not shadow the real reference modules
    for name in list(sys.modules):
        if name == "packnet_sfm" or name.startswith("packnet_sfm."):
            mod = sys.modules[name]
            if getattr(mod, "__pn_b200_dropin__", False):
                del sys.modules[name]
