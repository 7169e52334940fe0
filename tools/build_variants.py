#!/usr/bin/env python3
"""Build experiment variants of libacq_b200.so next to the product library (flydog_sdr_gps_b200/csrc/variants/).

    python tools/build_variants.py                 every named variant of flydog_sdr_gps_b200/_build.py VARIANTS
    python tools/build_variants.py l1_cta e1b_cta  the named ones
    python tools/build_variants.py name=DEF1,DEF2  an ad-hoc variant with the given -D defines (name= alone: none)
"""
import concurrent.futures as cf
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from flydog_sdr_gps_b200 import _build


def one(arg):
    name, eq, defs = arg.partition("=")
    if eq:
        return _build.build(defines=[x for x in defs.split(",") if x], out=_build.variant_path(name))
    return _build.build_variant(name, force=True)


if __name__ == "__main__":
    os.makedirs(os.path.join(_build.CSRC, "variants"), exist_ok=True)
    names = sys.argv[1:] or list(_build.VARIANTS)
    with cf.ThreadPoolExecutor(max_workers=min(len(names), os.cpu_count() or 1)) as ex:
        for path in ex.map(one, names):
            print(path)
