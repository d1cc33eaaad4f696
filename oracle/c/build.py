"""Builds oracle/c/libpgbp_oracle.so (gcc -O2 -march=native -fopenmp).  Test infrastructure.
The library is rebuilt when the source is newer OR when it was built on a different CPU model
(-march=native code must not travel between hosts).  When the source tree is read-only, the library
is built in a private cache directory of the user instead, under a name that hashes the source, the
compiler flags and the CPU model, so that no other source's build can be picked up."""
import hashlib
import os
import stat
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "pgbp_oracle.c")
LIB = os.path.join(HERE, "libpgbp_oracle.so")
LIBQ = os.path.join(HERE, "libpgbp_oracle_quad.so")  # same source in IEEE binary128 (-DPGBPO_QUAD, libquadmath)
TAG = LIB + ".host"
FLAGS = ["-O2", "-march=native", "-fopenmp", "-fPIC", "-shared", "-std=gnu11", "-ffp-contract=off"]


def _host():
    try:
        txt = open("/proc/cpuinfo").read()
        keep = [l for l in txt.splitlines() if l.startswith(("model name", "flags"))][:2]
        return hashlib.sha1("\n".join(keep).encode()).hexdigest()
    except OSError:
        return "unknown"


def _stale(lib, host):
    tag = lib + ".host"
    return (not os.path.exists(lib) or os.path.getmtime(lib) < os.path.getmtime(SRC)
            or not os.path.exists(tag) or open(tag).read().strip() != host)


def _compile(out, quad):
    extra = ["-DPGBPO_QUAD"] if quad else []
    subprocess.run(["gcc"] + FLAGS + extra + ["-o", out, SRC, "-lm"] + (["-lquadmath"] if quad else []), check=True)


def _private_dir():
    """<tmp>/pgbp_oracle-<uid> when it is a directory of this user that nobody else may read or write; otherwise
    a fresh directory from mkdtemp."""
    d = os.path.join(tempfile.gettempdir(), "pgbp_oracle-%d" % os.getuid())
    try:
        os.mkdir(d, 0o700)
    except FileExistsError:
        pass
    st = os.lstat(d)
    if not stat.S_ISDIR(st.st_mode) or st.st_uid != os.getuid() or st.st_mode & 0o077:
        return tempfile.mkdtemp(prefix="pgbp_oracle-")
    return d


def build(force=False, quad=False):
    host = _host()
    lib = LIBQ if quad else LIB
    if os.access(HERE, os.W_OK):
        if force or _stale(lib, host):
            _compile(lib, quad)
            open(lib + ".host", "w").write(host)
        return lib
    if not force and not _stale(lib, host):
        return lib
    # read-only tree: everything the library depends on goes into its name
    h = hashlib.sha1(open(SRC, "rb").read())
    h.update("\0".join(FLAGS + [str(quad), host]).encode())
    d = _private_dir()
    cached = os.path.join(d, "%s-%s.so" % (os.path.splitext(os.path.basename(lib))[0], h.hexdigest()))
    if force or not os.path.exists(cached):
        # compiled under a name of its own, then renamed: a process that has the library loaded keeps its copy
        fd, tmp = tempfile.mkstemp(suffix=".so", dir=d)
        os.close(fd)
        try:
            _compile(tmp, quad)
            os.replace(tmp, cached)
        finally:
            if os.path.exists(tmp):
                os.remove(tmp)
    return cached


if __name__ == "__main__":
    print(build(force=True))
    print(build(force=True, quad=True))
