"""Recipe for ``oracle/_ref/`` (build output, not in git): the original VMAS project, compiled to bytecode.

Two tests run the original project's own files: its scenario files on this package next to the original
(tests/test_reference_scenarios_dropin.py) and through the device-reset path (tests/test_reset_host_path.py).
:func:`build` (called by ``__graft_entry__.build``) compiles the original's ``vmas`` package from a checkout
into ``oracle/_ref/vmas/`` as sourceless ``.pyc`` files (its data files copied beside them), so that those
tests run wherever the build output goes, without the checkout.  Where no checkout is found, an existing
``oracle/_ref/`` is left as it is.
"""
import os
import py_compile
import shutil

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref")


def checkout():
    """The original project's checkout: ``$VMAS_REF``, else where it is kept on the build machines."""
    for path in (os.environ.get("VMAS_REF"), "/root/reference"):
        if path and os.path.isdir(os.path.join(path, "vmas")):
            return path
    return None


def build():
    """Returns ``oracle/_ref``, or None if there is neither a checkout nor an earlier build."""
    src = checkout()
    if src is None:
        return OUT if os.path.isdir(os.path.join(OUT, "vmas")) else None
    tmp = OUT + ".tmp"
    shutil.rmtree(tmp, ignore_errors=True)
    root = os.path.join(src, "vmas")
    for dirpath, dirnames, filenames in os.walk(root):
        dirnames[:] = sorted(d for d in dirnames if d != "__pycache__")
        dest = os.path.join(tmp, "vmas", os.path.relpath(dirpath, root))
        os.makedirs(dest, exist_ok=True)
        for name in sorted(filenames):
            path = os.path.join(dirpath, name)
            if name.endswith(".py"):
                py_compile.compile(path, cfile=os.path.join(dest, name[: -len(".py")] + ".pyc"), doraise=True)
            elif not name.endswith(".pyc"):
                shutil.copyfile(path, os.path.join(dest, name))
    shutil.rmtree(OUT, ignore_errors=True)
    os.replace(tmp, OUT)
    return OUT
