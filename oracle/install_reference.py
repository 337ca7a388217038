"""Install the unmodified reference package (lucidrains/glom-pytorch, pure Python) into ``oracle/_ref`` so that
``bench.py --impl reference`` and bench.py's cpu_baseline time the reference's own torch CPU forward.

The source is the checkout named by ``$GLOM_REF_PATH``, by default ``/root/reference``.  The package is pure Python
(``setup.py``: ``find_packages()`` = ``glom_pytorch/``), so installing it is copying that package unmodified; no pip
is needed.  ``oracle/_ref`` is a build product (git-ignored); no reference source is copied into the repository.

    GLOM_REF_PATH=<checkout> python -m oracle.install_reference
"""
import os
import shutil
import stat
import sys
import tempfile

TARGET = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")
DEFAULT_SOURCE = "/root/reference"
PACKAGE = "glom_pytorch"


def install(source=None, target=TARGET):
    """Returns (installed, where): installed is True when ``target/glom_pytorch`` exists (now or from an earlier
    call); `where` names the source, or says why nothing was installed."""
    if os.path.isfile(os.path.join(target, PACKAGE, "__init__.py")):
        return True, target
    source = source or os.environ.get("GLOM_REF_PATH") or DEFAULT_SOURCE
    pkg = os.path.join(source, PACKAGE)
    if not os.path.isfile(os.path.join(pkg, "__init__.py")):
        return False, f"no reference package at {pkg} (set $GLOM_REF_PATH to a glom-pytorch checkout)"
    os.makedirs(target, exist_ok=True)
    tmp = tempfile.mkdtemp(prefix=".install_", dir=target)
    try:
        staged = os.path.join(tmp, PACKAGE)
        shutil.copytree(pkg, staged, ignore=shutil.ignore_patterns("__pycache__", "*.pyc"))
        for d, _, files in os.walk(staged):            # copytree keeps the checkout's read-only modes
            for p in [d] + [os.path.join(d, f) for f in files]:
                os.chmod(p, os.stat(p).st_mode | stat.S_IWUSR)
        os.replace(staged, os.path.join(target, PACKAGE))   # a partial copy is never visible as installed
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return True, source


if __name__ == "__main__":
    ok, where = install()
    print(("installed from " if ok else "not installed: ") + where)
    sys.exit(0 if ok else 1)
