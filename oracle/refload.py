"""TEST INFRASTRUCTURE ONLY -- load the *unmodified* reference modules on top of the oracle shim.

Only usable where an unmodified checkout of the reference project is present: at ``oracle/_ref`` (ignored by git) or at the
directory named by ``MATRIX0_REFERENCE_ROOT``.  Used by
``tests/golden/make_golden.py`` to generate the committed golden vectors and by the ``not gpu``
pinning tests that compare ``oracle/*_ref.py`` restatements with the real reference code.

The reference's ``azchess/__init__.py`` and ``azchess/utils/__init__.py`` eagerly import the
orchestrator, arena, data manager etc. (``azchess/__init__.py:11-12``), which need packages that
are not installed.  We therefore register *empty* package objects named ``azchess`` and
``azchess.utils`` whose ``__path__`` points into the reference tree, so that
``importlib.import_module("azchess.mcts")`` executes ``azchess/mcts.py`` itself byte-for-byte
(with its relative imports resolving to the reference's ``encoding.py`` / ``utils/tensor.py``)
without running either ``__init__``.
"""
from __future__ import annotations

import importlib
import os
import sys
import types

_ORACLE_DIR = os.path.dirname(os.path.abspath(__file__))
REFERENCE_ROOT = os.environ.get("MATRIX0_REFERENCE_ROOT", os.path.join(_ORACLE_DIR, "_ref"))
MISSING = "needs the unmodified reference tree (oracle/_ref or MATRIX0_REFERENCE_ROOT)"


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "azchess", "mcts.py"))


def install_chess_shim() -> types.ModuleType:
    """Make ``import chess`` resolve to ``oracle/chess`` (unless real python-chess is importable)."""
    if "chess" in sys.modules:
        return sys.modules["chess"]
    if _ORACLE_DIR not in sys.path:
        sys.path.insert(0, _ORACLE_DIR)
    import chess  # noqa: F401  (oracle/chess)
    import chess.pgn  # noqa: F401
    import chess.polyglot  # noqa: F401
    import chess.syzygy  # noqa: F401
    return sys.modules["chess"]


def _stub_package(name: str, path: str) -> types.ModuleType:
    mod = sys.modules.get(name)
    if mod is None:
        mod = types.ModuleType(name)
        mod.__path__ = [path]  # type: ignore[attr-defined]
        mod.__package__ = name
        sys.modules[name] = mod
    return mod


def load_reference(*modules: str):
    """Import reference modules (e.g. ``"encoding"``, ``"mcts"``, ``"model.resnet"``) unmodified."""
    if not reference_available():
        raise FileNotFoundError(f"reference tree not found at {REFERENCE_ROOT}")
    install_chess_shim()
    az = os.path.join(REFERENCE_ROOT, "azchess")
    _stub_package("azchess", az)
    _stub_package("azchess.utils", os.path.join(az, "utils"))
    _stub_package("azchess.model", os.path.join(az, "model"))
    out = [importlib.import_module("azchess." + m) for m in modules]
    return out[0] if len(out) == 1 else out
