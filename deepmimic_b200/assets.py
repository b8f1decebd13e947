"""Asset root resolution.  DeepMimic arg files name assets relative to the directory that contains
data/ and args/ (the reference's repository root).  Order: $DEEPMIMIC_ASSET_ROOT, a checkout of the reference
named by $DEEPMIMIC_REFERENCE_ROOT (unless prefer_archive), else the archive tests/golden/assets.tar.gz unpacked once
next to it -- or, when the source tree is read-only, into a private temporary directory removed at exit."""
import atexit
import os
import shutil
import tarfile
import tempfile
import threading
import warnings

_lock = threading.Lock()
_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_tmp_root = None


def reference_root():
    """Root of a checkout of the original DeepMimic repository ($DEEPMIMIC_REFERENCE_ROOT), or None.  Only the checks
    against the reference's pretrained TF checkpoints need one; everything else runs on the committed archive."""
    ref = os.environ.get("DEEPMIMIC_REFERENCE_ROOT")
    return ref if ref and os.path.isdir(os.path.join(ref, "data", "characters")) else None


def _unpack(arc, out):
    os.makedirs(out, exist_ok=True)
    with tarfile.open(arc, "r:gz") as tf:
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            tf.extractall(out)
    open(os.path.join(out, ".unpacked"), "w").close()


def asset_root(prefer_archive: bool = False) -> str:
    global _tmp_root
    env = os.environ.get("DEEPMIMIC_ASSET_ROOT")
    if env:
        return env
    if not prefer_archive and reference_root():
        return reference_root()
    arc = os.path.join(_REPO, "tests", "golden", "assets.tar.gz")
    out = os.path.join(_REPO, "tests", "golden", "_assets")
    with _lock:
        stamp = os.path.join(out, ".unpacked")
        if os.path.exists(stamp) and os.path.getmtime(stamp) >= os.path.getmtime(arc):
            return out
        if _tmp_root is not None:
            return _tmp_root
        try:
            _unpack(arc, out)
            return out
        except OSError:          # read-only tree: unpack for this process only
            _tmp_root = tempfile.mkdtemp(prefix="deepmimic_b200_assets_")
            atexit.register(shutil.rmtree, _tmp_root, True)
            _unpack(arc, _tmp_root)
            return _tmp_root
