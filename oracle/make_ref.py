#!/usr/bin/env python
"""Recipe: stage the UNMODIFIED reference (gentaiscool/end2end-asr-pytorch) under oracle/_ref/ so it travels to the GPU box.

    python oracle/make_ref.py            # build container only: /root/reference -> oracle/_ref/

TEST INFRASTRUCTURE ONLY.  The reference is a pure-Python application (no setup.py, nothing to compile): "building" it
is copying the three packages the hot path imports -- models/, utils/, trainer/ (+ data/labels/*.json for the vocabularies)
-- byte for byte from where they lie under /root/reference.  oracle/_ref/ is listed in .gitignore (the sources never enter
this repository's history) and is NOT in .gpurunignore, so the `gpurun` snapshot carries it to the box, where
  * tests/test_host_logic.py::test_install_rebinds_reference_classes_and_keeps_module_tree binds b200asr.install() onto
    the unmodified reference classes (tests/test_gpu_reference.py compares with stored reference results instead),
  * bench.py --impl reference times the reference's own CPU path, and bench.py's `reference_gpu` object times the
    reference eager on the same B200.
Nothing in the product package imports from here.  `__graft_entry__.build()` calls stage() when /root/reference exists.
"""
import filecmp
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.environ.get("B200ASR_REFERENCE_SRC", "/root/reference")
DST = os.path.join(HERE, "_ref")
PARTS = ["models", "utils", "trainer", os.path.join("data", "labels")]
FILES = [os.path.join("data", "__init__.py"), os.path.join("data", "helper.py")]     # utils/metrics.py:7 imports data.helper


def stage(verbose=True):
    """Copy PARTS of SRC into oracle/_ref/ (idempotent).  Returns the number of files staged, 0 if SRC is absent."""
    if not os.path.isdir(os.path.join(SRC, "models", "asr")):
        if verbose:
            print(f"make_ref: {SRC} not present (GPU box): keeping the prebuilt oracle/_ref as is")
        return 0
    n = 0
    for part in PARTS:
        for root, dirs, files in os.walk(os.path.join(SRC, part)):
            dirs[:] = [d for d in dirs if d != "__pycache__"]
            rel = os.path.relpath(root, SRC)
            os.makedirs(os.path.join(DST, rel), exist_ok=True)
            for f in files:
                if not f.endswith((".py", ".json")):
                    continue
                s, d = os.path.join(root, f), os.path.join(DST, rel, f)
                if not (os.path.exists(d) and filecmp.cmp(s, d, shallow=False)):
                    shutil.copyfile(s, d)
                n += 1
    for rel in FILES:
        s, d = os.path.join(SRC, rel), os.path.join(DST, rel)
        if os.path.exists(s):
            os.makedirs(os.path.dirname(d), exist_ok=True)
            if not (os.path.exists(d) and filecmp.cmp(s, d, shallow=False)):
                shutil.copyfile(s, d)
            n += 1
        elif rel.endswith("__init__.py"):
            os.makedirs(os.path.dirname(d), exist_ok=True)
            open(d, "a").close()                      # namespace marker only (the reference has no data/__init__.py)
    if verbose:
        print(f"make_ref: {n} files of the unmodified reference staged in {DST}")
    return n


if __name__ == "__main__":
    sys.exit(0 if stage() >= 0 else 1)
