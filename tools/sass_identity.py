"""Compare the SASS of every kernel in two builds of the same object files.

    python tools/sass_identity.py OLD_DIR NEW_DIR [name.o ...]

Each object is disassembled with ``cuobjdump -sass`` and split into functions.  A function of OLD_DIR must have
identical instructions in NEW_DIR (addresses and encodings included, runs of blanks compared as one); functions only NEW_DIR has are listed as added.
Exits 1 when a function of OLD_DIR changed or disappeared.
"""
from __future__ import annotations

import os
import re
import subprocess
import sys


def functions(obj):
    text = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
    out, name = {}, None
    for line in text.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = m.group(1)
            out[name] = []
        elif name is not None and line.strip():
            out[name].append(" ".join(line.split()))  # (cuobjdump pads columns to the file's longest name)
    return out


def main(argv):
    old_dir, new_dir = argv[0], argv[1]
    names = argv[2:] or sorted(f for f in os.listdir(old_dir) if f.endswith(".o"))
    bad = 0
    for name in names:
        old, new = functions(os.path.join(old_dir, name)), functions(os.path.join(new_dir, name))
        same = [f for f in old if new.get(f) == old[f]]
        changed = [f for f in old if f in new and new[f] != old[f]]
        gone = [f for f in old if f not in new]
        added = [f for f in new if f not in old]
        print(f"{name}: {len(same)} of {len(old)} functions identical, {len(changed)} changed, {len(gone)} missing, "
              f"{len(added)} added")
        for f in changed:
            print(f"  CHANGED {f}")
        for f in gone:
            print(f"  MISSING {f}")
        for f in added:
            print(f"  added   {f}")
        bad += len(changed) + len(gone)
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
