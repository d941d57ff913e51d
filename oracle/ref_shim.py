"""Import shims that let the UNMODIFIED reference (pyDcop) import under Python 3.12 / numpy 2.
TEST INFRASTRUCTURE ONLY.

Only the golden generators under oracle/, the tests that run the reference and bench.py's
`reference-threadmode` baseline use this; nothing in the product path imports it.  The reference is
the copy oracle/install_reference.py installed into oracle/_ref/ (git-ignored, built by
__graft_entry__.build()), else its source tree (PYDCOP_REFERENCE); the tests that need it skip
where neither exists.

Shims (SURVEY.md §8c):
  1. collections.Iterable/Mapping/... aliases (reference: pydcop/dcop/yamldcop.py:32, dcop.py:238)
  2. stub `websocket_server` package (reference: pydcop/infrastructure/ui.py:36)
  3. stub `pulp` package (reference: ILP distributions, commands/generators/iot.py:47-49)
"""
import collections
import collections.abc
import os
import sys
import types

import install_reference

#: the unmodified reference: the installed copy in oracle/_ref/, else the source tree it is installed from
INSTALLED_ROOT = install_reference.TARGET
REFERENCE_ROOT = INSTALLED_ROOT if install_reference.installed() else install_reference.SOURCE


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "pydcop"))


def install() -> None:
    if not reference_available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    for n in ("Iterable", "Mapping", "Callable", "Sized", "MutableMapping", "Sequence",
              "Hashable", "Container", "Set", "MutableSet", "MutableSequence"):
        if not hasattr(collections, n):
            setattr(collections, n, getattr(collections.abc, n))
    if "websocket_server" not in sys.modules:
        ws = types.ModuleType("websocket_server")
        ws2 = types.ModuleType("websocket_server.websocket_server")
        ws2.WebsocketServer = type(
            "WebsocketServer", (), {"__init__": lambda self, *a, **k: None})
        ws.websocket_server = ws2
        sys.modules["websocket_server"] = ws
        sys.modules["websocket_server.websocket_server"] = ws2
    if "pulp" not in sys.modules:
        class _Stub(types.ModuleType):
            def __getattr__(self, n):
                if n.startswith("__"):
                    raise AttributeError(n)
                return object
        for name in ("pulp", "pulp.constants", "pulp.pulp", "pulp.solvers"):
            sys.modules[name] = _Stub(name)
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
