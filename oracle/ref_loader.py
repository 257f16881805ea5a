"""Import the UNMODIFIED reference modules from the reference checkout (MEGREADER_REFERENCE).

The reference's third-party deps (tensorboardX, apex, anyconfig, ...) are not installed, so
stub modules are injected into sys.modules first.  Only oracle/make_golden.py imports this
file, to record tests/golden/* (committed): no test, smoke() or bench.py needs the reference.
"""
import importlib
import os
import sys
import types

REF = os.environ.get("MEGREADER_REFERENCE", "/root/reference")

_STUBS = ["tensorboardX", "apex", "apex.parallel", "anyconfig", "munch", "editdistance", "imgaug",
          "imgaug.augmenters", "shapely", "shapely.geometry", "lmdb", "redis", "pyclipper", "gevent",
          "gevent.pywsgi", "geventwebsocket", "geventwebsocket.handler", "hanziconv", "flask", "boto3",
          "ipdb", "fire", "nori2", "Polygon"]


def available():
    return os.path.isdir(os.path.join(REF, "decoders"))


class _Anything:
    def __init__(self, *a, **k):
        pass

    def __call__(self, *a, **k):
        return _Anything()

    def __getattr__(self, name):
        return _Anything()


def _stub(name):
    m = types.ModuleType(name)
    m.__path__ = []
    m.__file__ = "<stub %s>" % name

    def _getattr(attr):
        if attr.startswith("__"):
            raise AttributeError(attr)
        return _Anything
    m.__getattr__ = _getattr
    return m


def install():
    """Put /root/reference on sys.path with stubbed third-party deps.  Returns True if usable."""
    if not available():
        return False
    import torch  # noqa: F401  (must be imported before any stub is visible)
    import torchvision  # noqa: F401
    for name in _STUBS:
        if name not in sys.modules:
            try:
                importlib.import_module(name)
            except Exception:
                sys.modules[name] = _stub(name)
    if REF not in sys.path:
        sys.path.insert(0, REF)
    return True


def load(modname):
    """e.g. load('decoders.ctc_loss2d')"""
    if not install():
        raise RuntimeError("reference not present at %s" % REF)
    return importlib.import_module(modname)
