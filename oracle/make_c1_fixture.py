#!/usr/bin/env python
"""Build tests/golden_large/c1_frames.tar.gz: config C1 (BASELINE.json configs[0]) = the reference's bundled Mg-TFSI/DME
trajectory, all 101 frames, reduced to the columns the parity tests read (id type x y z xu yu zu; the number tokens are
copied verbatim, so every parsed float is the one the reference parses from the original files).

The archive is ~20 MB and therefore NOT committed (tests/golden_large/ is git-ignored); the tests that need it skip when
it is absent.  Build it from a checkout of the reference project with
    MDPROP_REFERENCE_ROOT=<reference checkout> python oracle/make_c1_fixture.py
The known answers it is checked against (SURVEY.md 8c) were produced by the unmodified reference on the original files.
"""
import glob
import io
import os
import re
import sys
import tarfile

SRC = os.path.join(os.environ.get("MDPROP_REFERENCE_ROOT", ""), "data", "mg_tfsi_dme")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DST = os.path.join(ROOT, "tests", "golden_large", "c1_frames.tar.gz")
KEEP = ["id", "type", "x", "y", "z", "xu", "yu", "zu"]


def reduce_frame(text: str) -> str:
    lines = text.split("\n")
    k = next(i for i, ln in enumerate(lines) if ln.startswith("ITEM: ATOMS"))
    cols = lines[k].split()[2:]
    idx = [cols.index(c) for c in KEEP]
    out = lines[:k] + ["ITEM: ATOMS " + " ".join(KEEP)]
    for ln in lines[k + 1:]:
        t = ln.split()
        if t:
            out.append(" ".join(t[i] for i in idx))
    return "\n".join(out) + "\n"


def main():
    files = sorted(glob.glob(os.path.join(SRC, "dump.nvt.*.dump")), key=lambda f: int(re.findall(r"(\d+)\.dump$", f)[0]))
    if not files:
        sys.exit(f"no dump files under {SRC}")
    os.makedirs(os.path.dirname(DST), exist_ok=True)
    with tarfile.open(DST, "w:gz", compresslevel=6) as tar:
        for f in files:
            data = reduce_frame(open(f).read()).encode()
            ti = tarfile.TarInfo(os.path.basename(f))
            ti.size = len(data)
            tar.addfile(ti, io.BytesIO(data))
    print(DST, os.path.getsize(DST) // 1024, "KiB,", len(files), "frames")


if __name__ == "__main__":
    main()
