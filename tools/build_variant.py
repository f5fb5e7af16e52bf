#!/usr/bin/env python
"""Build a kernel-variant copy of libqlb.so (experiments only): tools/build_variant.py NAME -DQLB_X=1 ...
The library lands in quadruped_locomotion_b200/variants/libqlb_NAME.so; select it with QLB_LIB=<path>."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from quadruped_locomotion_b200 import build as qb  # noqa: E402


def main():
    name, flags = sys.argv[1], sys.argv[2:]
    out = os.path.join(qb.PKG, "variants", f"libqlb_{name}.so")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    print(qb.build(force=True, extra=flags, out=out))


if __name__ == "__main__":
    main()
