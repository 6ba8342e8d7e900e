"""TEST INFRASTRUCTURE ONLY -- make ``import chess`` resolve to the oracle restatement.

If the real python-chess is installed it wins (then the oracle restatements are checked against
the genuine third-party implementation); otherwise ``oracle/chess`` is registered under the name
``chess`` so that both the oracle modules and -- where the reference tree is present -- the unmodified
reference modules import it.
"""
import importlib.util
import os
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))

if "chess" not in sys.modules:
    _real = None
    try:
        _spec = importlib.util.find_spec("chess")
        if _spec is not None and _spec.origin and not os.path.abspath(_spec.origin).startswith(_HERE):
            _real = _spec
    except (ImportError, ValueError):
        _real = None
    if _real is None and _HERE not in sys.path:
        sys.path.insert(0, _HERE)
    import chess  # noqa: F401,E402
    try:
        import chess.pgn  # noqa: F401,E402
    except ImportError:
        pass

USING_ORACLE_SHIM = os.path.abspath(getattr(sys.modules["chess"], "__file__", "")).startswith(_HERE)
