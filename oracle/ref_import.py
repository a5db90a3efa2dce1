"""Import the real reference: from its source tree (CZ_REFERENCE_ROOT) when that is present, else from the
byte-compiled modules `oracle/build_ref.py` wrote into oracle/_ref (sourceless imports of the same code).

Used only to validate the restatements in this directory and to generate tests/golden/; callers must handle
`available() == False`.  The generators also read the reference's data files and need `source_available()`.
Recipe from SURVEY.md Appendix B: PYTHONPATH root + the package dir itself (config.py does
`import configs.mini`), data/log dirs redirected to a scratch directory.
"""
import os
import sys
import tempfile

REF_ROOT = os.environ.get("CZ_REFERENCE_ROOT", "/root/reference")


REF_BUILD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")


def source_available():
    return os.path.isdir(os.path.join(REF_ROOT, "cchess_alphazero", "environment"))


def build_available():
    return os.path.exists(os.path.join(REF_BUILD, "cchess_alphazero", "environment", "static_env.pyc"))


def available():
    return source_available() or build_available()


def import_root():
    return REF_ROOT if source_available() else REF_BUILD


_done = False


def setup():
    global _done
    if _done:
        return
    if not available():
        raise RuntimeError("reference not present: neither its source tree nor oracle/_ref")
    sys.dont_write_bytecode = True
    scratch = tempfile.mkdtemp(prefix="cz_ref_")
    os.environ.setdefault("PROJECT_DIR", scratch)
    os.environ.setdefault("DATA_DIR", os.path.join(scratch, "data"))
    root = import_root()
    for p in (root, os.path.join(root, "cchess_alphazero")):
        if p not in sys.path:
            sys.path.insert(0, p)
    _done = True


def senv():
    setup()
    import cchess_alphazero.environment.static_env as m
    return m


def lookup_tables():
    setup()
    import cchess_alphazero.environment.lookup_tables as m
    return m


def player_module():
    setup()
    import cchess_alphazero.agent.player as m
    return m


def config(kind="mini"):
    setup()
    from cchess_alphazero.config import Config
    return Config(kind)
