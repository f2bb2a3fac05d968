"""Compare the SASS of every kernel of two builds of the library (no GPU needed).

    python tools/scripts/sass_diff.py OLD.so NEW.so [--out FILE.json]

`cuobjdump -sass` of both libraries is split per kernel (mangled name); a kernel of OLD is unchanged when NEW has a
kernel of the same name with the same instructions (addresses and the line-info comments dropped).  Prints and
optionally writes the kernels of OLD that are missing or changed in NEW and the kernels NEW adds; exit status 1 when
any kernel of OLD changed or disappeared."""
from __future__ import annotations

import argparse
import json
import re
import subprocess
import sys


def kernels(lib: str) -> dict[str, str]:
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    res, name, body = {}, None, []
    for ln in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", ln)
        if m:
            if name:
                res[name] = "\n".join(body)
            name, body = m.group(1), []
            continue
        if name is None:
            continue
        ins = re.match(r"\s*/\*[0-9a-f]+\*/\s*(.*?);", ln)
        if ins:
            body.append(ins.group(1).strip())
    if name:
        res[name] = "\n".join(body)
    return res


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    old, new = kernels(a.old), kernels(a.new)
    missing = sorted(k for k in old if k not in new)
    changed = sorted(k for k in old if k in new and old[k] != new[k])
    res = {"old_kernels": len(old), "new_kernels": len(new), "unchanged": len(old) - len(missing) - len(changed),
           "missing": missing, "changed": changed, "added": sorted(k for k in new if k not in old)}
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))
    return 1 if missing or changed else 0


if __name__ == "__main__":
    sys.exit(main())
