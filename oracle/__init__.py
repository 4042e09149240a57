"""TEST INFRASTRUCTURE ONLY: CPU restatement ("oracle") of the reference's algorithm for the hot
path.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import anything from here; the product package trinerflet_b200 never does."""
import os


def reference_path(*parts):
    """<checkout of the original TriNerfLet project>/<parts>, the checkout named by the environment variable
    TRINERFLET_REFERENCE; "" when that is not set.  Only the live comparisons with the original read it (tests that skip
    without it, the golden-fixture generators, the build of its CUDA extensions as a checker)."""
    root = os.environ.get("TRINERFLET_REFERENCE", "")
    return os.path.join(root, *parts) if root else ""


def require_reference(path):
    """`path` (from reference_path) if it is a directory; otherwise an error that says what to set."""
    if not os.path.isdir(path):
        raise RuntimeError("set TRINERFLET_REFERENCE to a checkout of the original TriNerfLet project"
                           + (f" ({path} is not a directory)" if path else ""))
    return path
