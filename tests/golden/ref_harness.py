"""
Import the (Python) reference, an unmodified EVcouplings checkout whose directory is given by the
EVCOUPLINGS_REFERENCE environment variable (or set_root()).

The reference's optional plotting / batch dependencies may be absent
(ruamel.yaml, matplotlib, seaborn, bokeh, billiard, Bio); none of them is on
the couplings path, so they are shimmed (SURVEY.md Appendix B).  Used only by
tests/golden/make_golden.py (golden-vector generation); the tests read the
fixtures it writes and never import the reference.
"""
import importlib.abc
import importlib.machinery
import os
import sys
import types
import warnings
from unittest import mock

REFERENCE_ROOT = os.environ.get("EVCOUPLINGS_REFERENCE", "")
_STUB_ROOTS = ("matplotlib", "seaborn", "bokeh", "billiard", "Bio", "mpl_toolkits")


def set_root(path):
    global REFERENCE_ROOT
    REFERENCE_ROOT = os.path.abspath(path)


def available():
    return bool(REFERENCE_ROOT) and os.path.isdir(os.path.join(REFERENCE_ROOT, "evcouplings"))


class _StubLoader(importlib.abc.Loader):
    def create_module(self, spec):
        m = mock.MagicMock(name=spec.name)
        m.__name__ = spec.name
        m.__path__ = []
        m.__spec__ = spec
        m.__loader__ = self
        return m

    def exec_module(self, module):
        pass


class _StubFinder(importlib.abc.MetaPathFinder):
    def find_spec(self, fullname, path=None, target=None):
        if fullname.split(".")[0] in _STUB_ROOTS:
            return importlib.machinery.ModuleSpec(fullname, _StubLoader(), is_package=True)
        return None


def _install_ruamel_shim():
    try:
        import ruamel.yaml  # noqa: F401
        return
    except ImportError:
        pass
    import yaml
    ruamel = types.ModuleType("ruamel")
    ruamel.__path__ = []
    ry = types.ModuleType("ruamel.yaml")
    ry.__path__ = []
    ry.safe_load = yaml.safe_load
    ry.load = yaml.load
    ry.dump = yaml.dump
    ry.Dumper = yaml.Dumper
    ry.RoundTripLoader = yaml.SafeLoader
    ry.RoundTripDumper = yaml.Dumper
    ry.parser = yaml.parser
    ry.scanner = yaml.scanner
    comments = types.ModuleType("ruamel.yaml.comments")

    class CommentedBase(object):
        pass

    comments.CommentedBase = CommentedBase
    ry.comments = comments
    ruamel.yaml = ry
    sys.modules["ruamel"] = ruamel
    sys.modules["ruamel.yaml"] = ry
    sys.modules["ruamel.yaml.comments"] = comments


_installed = False


def install():
    """Make ``import evcouplings`` resolve to the unmodified reference."""
    global _installed
    if _installed:
        return
    if not available():
        raise RuntimeError("no EVcouplings checkout at %r (set EVCOUPLINGS_REFERENCE)" % REFERENCE_ROOT)
    warnings.filterwarnings("ignore", category=SyntaxWarning)
    _install_ruamel_shim()
    if not any(isinstance(f, _StubFinder) for f in sys.meta_path):
        sys.meta_path.append(_StubFinder())
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    _installed = True
