"""Copies the UNMODIFIED reference sources of the hot path (drqv2.py, utils.py, replay_buffer.py) from
the reference checkout (DRQ_REFERENCE, else BASELINE.json's reference_path /root/reference) into
baseline/_ref/ (git-ignored), so that `bench.py --impl reference` and the reference arm of bench.py
can time the reference's own implementation.  The reference is pure Python (nothing to compile);
hydra / omegaconf, which it imports but never uses on this path, are stubbed at import time by the
caller (SURVEY.md §8c).  Run by __graft_entry__.build(); a checkout that is absent, or that the
building user may not read, installs nothing."""
import os
import pathlib
import shutil
import sys

SRC = pathlib.Path(os.environ.get("DRQ_REFERENCE", "/root/reference"))
DST = pathlib.Path(__file__).resolve().parent / "_ref"
NAMES = ("drqv2.py", "utils.py", "replay_buffer.py")


def install():
    if not all(os.access(SRC / name, os.R_OK) for name in NAMES):   # absent, or not readable by this user
        return False
    DST.mkdir(parents=True, exist_ok=True)
    for name in NAMES:
        dst = DST / name
        if dst.exists():
            dst.chmod(0o644)
        shutil.copyfile(SRC / name, dst)
        dst.chmod(0o444)
    return True


if __name__ == "__main__":
    print("installed" if install() else "reference not present", file=sys.stderr)
