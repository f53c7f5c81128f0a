"""Import the UNMODIFIED reference package from /root/reference inside THIS container.

TEST INFRASTRUCTURE ONLY.  Used by the fixture generators (oracle/gen_golden*.py), whose
output under tests/golden/ is what the tests compare against; no test, smoke() or bench.py
calls it.

Shims (SURVEY.md section 8c): a stub `odtk._C` (the compiled extension is absent) and
`torchvision.models.{resnet,mobilenet}.model_urls` (removed in torchvision >= 0.13).
"""
import collections
import os
import sys
import types

REF_ROOT = os.environ.get("ODTK_REFERENCE", "/root/reference")


def available():
    return os.path.isdir(os.path.join(REF_ROOT, "odtk"))


def import_reference():
    """Returns the reference `odtk` package (box, model, loss importable)."""
    if "odtk" in sys.modules and getattr(sys.modules["odtk"], "__odtk_ref__", False):
        return sys.modules["odtk"]
    import torchvision.models.resnet as vrn
    import torchvision.models.mobilenet as vmn
    for m in (vrn, vmn):
        if not hasattr(m, "model_urls"):
            m.model_urls = collections.defaultdict(lambda: None)
    stub = types.ModuleType("odtk._C")

    def _absent(*a, **k):
        raise RuntimeError("odtk._C is a stub: the reference extension is not built here")

    stub.decode = stub.nms = stub.iou = _absent
    stub.Engine = type("Engine", (), {})
    sys.modules["odtk._C"] = stub
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    import odtk  # noqa: F401
    import odtk.box  # noqa: F401
    import odtk.loss  # noqa: F401
    import odtk.model  # noqa: F401
    odtk.__odtk_ref__ = True
    return odtk


def patched_cpu_decode():
    """The reference's CPU `box.decode` (odtk/box.py:255-309) with its three true divisions on
    index tensors (lines 291, 296-297: crash on torch >= 1.6) turned into floor divisions.
    The source text is read from /root/reference at call time and patched in memory."""
    import inspect
    odtk = import_reference()
    src = inspect.getsource(odtk.box.decode)
    src = src.replace("(indices / width / height) % num_classes", "(indices // width // height) % num_classes")
    src = src.replace("(indices / width) % height", "(indices // width) % height")
    src = src.replace("indices / num_classes / height / width", "indices // num_classes // height // width")
    ns = dict(vars(odtk.box))
    exec(compile(src, "<patched odtk.box.decode>", "exec"), ns)
    return ns["decode"]
