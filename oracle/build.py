"""Build recipe for the oracle's C restatement (test infrastructure).

`python -m oracle.build` compiles oracle/b2d_oracle.c into oracle/libb2d_oracle.so with gcc.
The reference itself (Rust + OpenGL) cannot be built here -- no rustc/cargo, crates not vendored,
no GL context -- so there is no oracle/_ref; DESIGN.md records this.

The library doubles as bench.py's CPU baseline, so it is compiled `-O3 -march=native` for the machine that
runs it: the host's CPU signature is recorded next to the .so and a library built on another machine (the
in-tree .so travels to the GPU box with the snapshot) is rebuilt there before it is loaded.
"""
import hashlib
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "b2d_oracle.c")
OUT = os.path.join(HERE, "libb2d_oracle.so")
HOST = OUT + ".host"
FLAGS = ["-O3", "-march=native", "-std=c11", "-fopenmp", "-fPIC", "-shared", "-fwrapv",
         "-Wall", "-Wextra", "-Wno-unused-parameter"]


def host_signature() -> str:
    """Model name + ISA flags of the first CPU (what -march=native keys on), hashed."""
    sig = []
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith(("model name", "flags")):
                    sig.append(line.split(":", 1)[1].strip())
                if len(sig) == 2:
                    break
    except OSError:
        pass
    return hashlib.sha256(("|".join(sig) + "|" + " ".join(FLAGS)).encode()).hexdigest()[:16]


def needs_build() -> bool:
    if not os.path.exists(OUT) or os.path.getmtime(OUT) < os.path.getmtime(SRC):
        return True
    try:
        with open(HOST) as f:
            return f.read().strip() != host_signature()
    except OSError:
        return True


def build(force: bool = False) -> str:
    if not force and not needs_build():
        return OUT
    if not os.access(HERE, os.W_OK):
        # a read-only tree whose library was built for another host: this host's build goes to a temporary directory
        out = os.path.join(tempfile.mkdtemp(prefix="b2d_oracle_"), os.path.basename(OUT))
        subprocess.check_call(["gcc"] + FLAGS + ["-o", out, SRC])
        return out
    subprocess.check_call(["gcc"] + FLAGS + ["-o", OUT, SRC])
    with open(HOST, "w") as f:
        f.write(host_signature() + "\n")
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv))
