"""ORACLE — test infrastructure only.  Build of oracle/osqp_admm.c into liboracle_osqp.so (make + gcc; no Python
dependencies, so that building the project needs none of the oracle's)."""
import hashlib
import os
import stat
import subprocess
import tempfile

_HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(_HERE, "_build", "liboracle_osqp.so")


def _stamp():
    """Content hash of the source, the build recipe and the host CPU (the library is built with -march=native and
    travels with the repo snapshot: a different host must rebuild it)."""
    h = hashlib.sha256()
    for f in ("osqp_admm.c", "Makefile"):
        h.update(open(os.path.join(_HERE, f), "rb").read())
    try:
        cpu = [l for l in open("/proc/cpuinfo") if l.startswith(("model name", "flags"))][:2]
    except OSError:
        cpu = []
    h.update("".join(cpu).encode())
    return h.hexdigest()


def _writable(d):
    while not os.path.exists(d):
        d = os.path.dirname(d)
    return os.access(d, os.W_OK)


def _private_dir(d):
    """d (created with mode 0700 if missing) when it is a directory of this user that no other user can write, else None:
    a library found in a shared directory is only loaded when no one else can have put it there."""
    try:
        os.mkdir(d, 0o700)
    except FileExistsError:
        pass
    except OSError:
        return None
    st = os.lstat(d)
    if stat.S_ISDIR(st.st_mode) and st.st_uid == os.getuid() and not st.st_mode & (stat.S_IWGRP | stat.S_IWOTH):
        return d
    return None


def _paths(d):
    return os.path.join(d, os.path.basename(SO)), os.path.join(d, "liboracle_osqp.sha256")


def _current(d, want):
    so, stamp = _paths(d)
    return os.path.exists(so) and os.path.exists(stamp) and open(stamp).read() == want


def build(force=False):
    """The library in oracle/_build, rebuilt when its stamp differs.  A stale library in a tree that cannot be written
    (a read-only checkout, built on another host) is rebuilt in a per-user temporary directory instead, or, when that
    directory is not private to this user, in a fresh one."""
    want = _stamp()
    d = os.path.dirname(SO)
    if not force and _current(d, want):
        return _paths(d)[0]
    if not _writable(d):
        d = _private_dir(os.path.join(tempfile.gettempdir(), "mpcb_oracle_%d_%s" % (os.getuid(), want[:16])))
        if d is not None and not force and _current(d, want):
            return _paths(d)[0]
        if d is None:
            d = tempfile.mkdtemp(prefix="mpcb_oracle_")
    so, stamp = _paths(d)
    subprocess.check_call(["make", "-s", "-B", "-C", _HERE, "OUT=" + d])
    open(stamp, "w").write(want)
    return so
