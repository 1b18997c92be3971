"""Writes tests/golden/flat_<world>.txt: what the C-ABI (rkFDChainRegFile / rkFDContactInfoScanFile + the flattening of
rkFDUpdateInit) makes of the reference's own example/model/*.ztk files, as text (`RkFD.describe_model()`).  The repository
does not contain the reference, so the tests load these tables (`chains.world_from_flat`); tests/test_capi_host.py checks,
when ROKIFD_REFERENCE names a reference tree, that they are what its files flatten to.  Run from the repo root:
    ROKIFD_REFERENCE=<path of a mi-lib/roki-fd checkout> python tests/golden/make_flat_models.py"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import rokifd_b200  # noqa: F401,E402
from test_capi_host import REF_WORLDS, reference_world_description  # noqa: E402

for name in REF_WORLDS:
    if name == "arm2dof_on_floor":
        continue
    desc = reference_world_description(name)
    with open(os.path.join(ROOT, "tests", "golden", "flat_%s.txt" % name), "w") as f:
        for k, v in desc.items():
            f.write("%s: %s\n" % (k, " ".join(repr(float(x)) for x in v)))
    print(name, "links %d dof %d vertices %d slots %d" % (desc["dims"][0], desc["dims"][1], desc["dims"][6], desc["dims"][5]))
