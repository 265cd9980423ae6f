"""Recipe for oracle/_ref: the UNMODIFIED reference files of the hot path, copied byte for byte from the read-only
checkout so that `bench.py --impl reference` can time the reference's OWN `WaveRNN.generate()` on the GPU box's host
cores (/root/reference does not exist there).  TEST / BENCH INFRASTRUCTURE ONLY.

    python oracle/make_ref.py            # also run by __graft_entry__.build() when /root/reference is present

oracle/_ref/ is git-ignored (reference sources never enter this repository's history) but NOT gpurun-ignored, so it
travels to the GPU box with the snapshot like a built .so.  The files are the closure of `import
models.fatchord_version` (fatchord_version.py:1-9): the model, utils/{__init__, display, dsp, distribution}.py and
hparams.py; a MANIFEST with their sha256 is written next to them and checked by bench.py before use.
"""
import hashlib
import json
import os
import shutil
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
SRC = Path(os.environ.get("WAVERNN_REFERENCE", "/root/reference"))
DST = HERE / "_ref"
FILES = ("models/__init__.py", "models/fatchord_version.py", "utils/__init__.py", "utils/display.py", "utils/dsp.py",
         "utils/distribution.py", "hparams.py", "LICENSE.txt")


def main() -> int:
    if not os.path.isfile(SRC / "models" / "fatchord_version.py"):      # False also where it cannot be read
        print(f"oracle/make_ref.py: no reference checkout at {SRC}; keeping whatever oracle/_ref already holds")
        return 0
    manifest = {}
    for rel in FILES:
        dst = DST / rel
        dst.parent.mkdir(parents=True, exist_ok=True)
        shutil.copyfile(SRC / rel, dst)
        os.chmod(dst, 0o644)
        manifest[rel] = hashlib.sha256(dst.read_bytes()).hexdigest()
    (DST / "MANIFEST.json").write_text(json.dumps({"source": str(SRC), "sha256": manifest}, indent=1))
    print(f"oracle/_ref: {len(FILES)} files copied from {SRC}")
    return 0


def verify() -> bool:
    """True when oracle/_ref holds exactly the files the manifest describes."""
    m = DST / "MANIFEST.json"
    if not m.is_file():
        return False
    try:
        want = json.loads(m.read_text())["sha256"]
        return all(hashlib.sha256((DST / rel).read_bytes()).hexdigest() == h for rel, h in want.items()) and \
            "models/fatchord_version.py" in want
    except Exception:
        return False


if __name__ == "__main__":
    sys.exit(main())
