"""TEST INFRASTRUCTURE ONLY.  Locate and import the *real*, unmodified reference.

Resolution order of the reference root:
  1. ``$SUPCON_REFERENCE_ROOT``
  2. ``/root/reference``            (the build container)
  3. ``oracle/_ref``                (verbatim copies staged by ``oracle/build_ref.py``; git-ignored, shipped
                                     with the gpurun snapshot -- this is what the GPU box sees)

Nothing under ``wav2vec_contr_loss_b200/`` imports this module.
"""
import importlib.util
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
STAGED_ROOT = os.path.join(_HERE, "_ref")


def reference_root():
    if os.environ.get("SUPCON_REFERENCE_DISABLE"):   # tests of the port fall-back
        return None
    for cand in (os.environ.get("SUPCON_REFERENCE_ROOT"), "/root/reference", STAGED_ROOT):
        if cand and os.path.isfile(os.path.join(cand, "loss.py")):
            return cand
    return None


REFERENCE_ROOT = reference_root() or "/root/reference"


def reference_available() -> bool:
    return reference_root() is not None


def reference_kind() -> str:
    """'source tree' (build container) or 'staged copy' (oracle/_ref on the GPU box)."""
    root = reference_root()
    if root is None:
        return "absent"
    return "staged copy" if os.path.abspath(root) == os.path.abspath(STAGED_ROOT) else "source tree"


def load_reference_module(name: str = "loss"):
    """Load ``<reference root>/<name>.py`` under a private module name so it can
    never shadow (or be shadowed by) the drop-in ``loss`` module of this repo."""
    root = reference_root()
    if root is None:
        raise FileNotFoundError("reference not found (neither /root/reference nor oracle/_ref)")
    path = os.path.join(root, name + ".py")
    if not os.path.isfile(path):
        raise FileNotFoundError(path)
    spec = importlib.util.spec_from_file_location("_reference_" + name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod
