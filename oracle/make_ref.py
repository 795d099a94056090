"""TEST / BASELINE INFRASTRUCTURE -- not imported by the product path.

Stages the UNMODIFIED reference package so that it can travel to the GPU box:

    python oracle/make_ref.py          # /root/reference/ratinabox/**/*.py  ->  oracle/_ref/ratinabox/

`oracle/_ref/` is git-ignored (reference sources never enter this repository's history) but NOT gpurun-ignored, exactly
like the built `.so`: `bench.py --impl reference`, `bench.py`'s `cpu_baseline` leg and
`tests/test_gpu_reference_binding.py` import the live reference from there through `oracle/ref_shim.py` (stand-ins for the
absent matplotlib / shapely).  Only Python sources are staged (the 7 MB of trajectory datasets under `ratinabox/data` are
not on the hot path); files are copied byte for byte and a manifest with their SHA-256 is written next to them.
`__graft_entry__.build()` runs this whenever /root/reference is present."""
import hashlib
import json
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.environ.get("RIAB_REFERENCE_ROOT", "/root/reference")
DST = os.path.join(HERE, "_ref")


def stage(verbose=True):
    pkg = os.path.join(SRC, "ratinabox")
    if not os.path.isdir(pkg):
        if verbose:
            print(f"[make_ref] {pkg} not present: nothing staged", file=sys.stderr)
        return None
    out = os.path.join(DST, "ratinabox")
    if os.path.isdir(out):
        shutil.rmtree(out)
    manifest = {}
    for root, dirs, files in os.walk(pkg):
        dirs[:] = [d for d in dirs if d not in ("data", "__pycache__", "TaskEnv_example_files")]
        for f in files:
            if not f.endswith(".py"):
                continue
            src = os.path.join(root, f)
            rel = os.path.relpath(src, SRC)
            dst = os.path.join(DST, rel)
            os.makedirs(os.path.dirname(dst), exist_ok=True)
            shutil.copyfile(src, dst)
            manifest[rel] = hashlib.sha256(open(src, "rb").read()).hexdigest()
    version = None
    try:
        for line in open(os.path.join(SRC, "setup.cfg")):
            if line.strip().startswith("version"):
                version = line.split("=")[1].strip()
    except OSError:
        pass
    json.dump({"source": SRC, "version": version, "files": manifest}, open(os.path.join(DST, "MANIFEST.json"), "w"), indent=1)
    if verbose:
        print(f"[make_ref] staged {len(manifest)} files of RatInABox {version} into {DST}", file=sys.stderr)
    return DST


if __name__ == "__main__":
    stage()
