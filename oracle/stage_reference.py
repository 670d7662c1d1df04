"""Stage the UNMODIFIED reference modules of the hot path into oracle/_ref/ (git-ignored).

TEST / MEASUREMENT INFRASTRUCTURE (oracle/).  When SSD_REFERENCE_ROOT names a checkout of the original project,
`__graft_entry__.build()` copies the reference's own files — byte for byte, nothing is edited — into `oracle/_ref/`, which
is listed in .gitignore (never committed) and can travel with a built tree to a machine without the checkout.  The only
consumer is `oracle/ref_bench.py` (bench.py's cpu_baseline / `--impl reference` arm): it times the reference's Python env
loop on the host cores.
"""
import os
import shutil

from . import ref_stubs

# what `utils/env_creator_functions.py:1-10` imports (the env classes, the wrapper, the contracts)
FILES = ["__init__.py", "LICENSE", "utils/__init__.py", "utils/env_creator_functions.py", "contract/contract.py", "contract/contract_list.py",
         "environments/__init__.py", "environments/Agent.py", "environments/map_env.py", "environments/env_utils.py",
         "environments/cleanup_new.py", "environments/harvest_new.py", "environments/cleanup_features.py",
         "environments/harvest_features.py", "environments/self_driving_car_accelerate.py", "environments/two_stage_train.py"]


def stage(src=ref_stubs.REFERENCE_ROOT, dst=ref_stubs.STAGED_ROOT):
    """Returns the staged root, or None when neither a reference checkout nor an earlier staged copy is present."""
    if not src or not os.path.isdir(os.path.join(src, "environments")):
        return dst if os.path.isdir(os.path.join(dst, "environments")) else None
    for rel in FILES:
        s = os.path.join(src, rel)
        if not os.path.exists(s):
            continue
        d = os.path.join(dst, rel)
        os.makedirs(os.path.dirname(d), exist_ok=True)
        shutil.copyfile(s, d)
    with open(os.path.join(dst, "STAGED_FROM"), "w") as f:
        f.write("unmodified copy of %s made by oracle/stage_reference.py; not part of this repository\n" % src)
    return dst


if __name__ == "__main__":
    print(stage())
