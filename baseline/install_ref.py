#!/usr/bin/env python
"""Install the UNMODIFIED reference's env path under baseline/_ref/ so that bench.py can time it on the host cores.

The reference (Nielsencu/primal-ppo) is a plain Python repo without packaging (there is nothing to `pip install`), so the
"install" is a verbatim copy of the modules the env path imports from a checkout of it (MAPF_REFERENCE_PATH).  Run it by
hand; baseline/_ref/ is git-ignored, so reference sources never enter this repo's history."""
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
DEST = os.path.join(HERE, "_ref")
SRC = os.environ.get("MAPF_REFERENCE_PATH", "/root/reference")
FILES = ["mapf_gym.py", "util.py", "alg_parameters.py", "map_generator.py", "astar_4.py", "astar_8.py"]


def install(force: bool = False) -> bool:
    if not os.path.isfile(os.path.join(SRC, "mapf_gym.py")):
        return os.path.isfile(os.path.join(DEST, "mapf_gym.py"))
    os.makedirs(DEST, exist_ok=True)
    for f in FILES:
        s, d = os.path.join(SRC, f), os.path.join(DEST, f)
        if force or not os.path.exists(d) or open(s, "rb").read() != open(d, "rb").read():
            shutil.copyfile(s, d)
    return True


if __name__ == "__main__":
    ok = install(force="-f" in sys.argv)
    print("baseline/_ref:", "installed" if ok else "reference not available")
