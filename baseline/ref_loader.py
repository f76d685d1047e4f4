"""Imports the UNMODIFIED reference (mapbox/robosat 1.2.0) from `oracle/_ref` for the benchmark's reference arm.

`oracle/_ref` is git-ignored; `__graft_entry__.build()` installs it with `oracle/build.sh` where the reference source is readable.

Nothing of the reference is changed; what is needed to import it without its optional dependencies (SURVEY.md Appendix A):
  * `mercantile` is absent           -> `baseline/shim/mercantile.py` (Tile namedtuple)
  * `robosat.utils` needs matplotlib -> a stub module with `plot()` (only `tools/train.py` imports it)
  * `resnet50(pretrained=True)` needs the network -> `robosat.unet.resnet50` is wrapped to pass pretrained=False; the weights
    come from the same seeded synthetic state_dict the GPU arm uses.
Bench / test infrastructure: the product package never imports this.
"""

import os
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.path.join(os.path.dirname(HERE), "oracle", "_ref")


def available():
    return os.path.exists(os.path.join(REF, "robosat", "unet.py"))


def load():
    """-> the reference's `robosat` package (modules `unet`, `losses`, `tools.predict` ... importable afterwards)"""
    if not available():
        raise ImportError("oracle/_ref is not installed (see oracle/build.sh)")
    for p in (os.path.join(HERE, "shim"), REF):
        if p not in sys.path:
            sys.path.insert(0, p)
    import robosat  # noqa: F401  (the reference package; this repo's package is `robosat_b200`)

    if "robosat.utils" not in sys.modules:
        fake = types.ModuleType("robosat.utils")
        fake.plot = lambda out, history: None
        sys.modules["robosat.utils"] = fake
    import robosat.unet as U

    if not getattr(U.resnet50, "_rsb_no_download", False):
        _orig = U.resnet50

        def resnet50(pretrained=True, **kw):
            return _orig(pretrained=False, **kw)

        resnet50._rsb_no_download = True
        U.resnet50 = resnet50
    return robosat


def reference_net(state_dict, num_classes):
    """The reference's model exactly as `rs predict` builds it on a GPU-less host (robosat/tools/predict.py:47-68):
    UNet(num_classes) wrapped in nn.DataParallel, weights from `state_dict`, eval mode, CPU."""
    import torch

    load()
    from robosat.unet import UNet

    net = torch.nn.DataParallel(UNet(num_classes))
    net.load_state_dict(state_dict)
    net.eval()
    return net
