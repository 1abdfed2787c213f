"""Compiles oracle/prophet_oracle.c (the plain-C restatement used as checker and CPU baseline)
into oracle/_build/libprophet_oracle.so with gcc.  Test infrastructure only."""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_build")
LIB = os.path.join(OUT, "libprophet_oracle.so")
SRC = os.path.join(HERE, "prophet_oracle.c")
CFLAGS = ["-O2", "-std=c11", "-fPIC", "-shared", "-fopenmp", "-fno-fast-math"]


def _digest() -> str:
    h = hashlib.sha256()
    with open(SRC, "rb") as f:
        h.update(f.read())
    h.update(" ".join(CFLAGS).encode())
    return h.hexdigest()


def build(force: bool = False) -> str:
    # up to date by content, not mtime: a copied tree (mtimes not kept) must not recompile, and may be read-only
    stamp = LIB + ".digest"
    digest = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == digest:
        return LIB
    os.makedirs(OUT, exist_ok=True)
    cmd = ["gcc", *CFLAGS, "-o", LIB, SRC, "-lm"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("gcc failed building the C oracle")
    with open(stamp, "w") as f:
        f.write(digest)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv))
