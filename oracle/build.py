"""oracle/build.py -- TEST INFRASTRUCTURE.  Compiles the C restatement (oracle/voxelize.c).

`oracle/_ref/` (a compile of the *reference's own* sources) is not produced:
the reference's arithmetic for this path lives in the third-party `spconv` /
`cumm` packages, which are absent from the reference repository (SURVEY.md fact 2),
so there is nothing of the reference to compile.  DESIGN.md records this.
"""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "liboracle_vox.so")
SRC = os.path.join(HERE, "voxelize.c")


def build(force: bool = False) -> str:
    if (not force) and os.path.exists(LIB) and os.path.getmtime(LIB) >= os.path.getmtime(SRC):
        return LIB
    cmd = ["gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC",
           "-o", LIB, SRC, "-lm"]
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force=True))
