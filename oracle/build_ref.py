"""Recipe for oracle/_ref/: the reference's own hot-path package, unmodified, where bench.py's CPU arm can import it.

TEST / MEASUREMENT INFRASTRUCTURE ONLY -- nothing under neko_b200/ imports it.

The GPU box has no /root/reference, and the reference cannot be pip-installed into a target directory: its setup.py
declares ``packages=['gato']`` only, so ``pip install --target ... /root/reference`` ships gato/__init__.py and none of
the sub-packages (tried: DESIGN.md section 1).  The reference is pure Python, so "building" it is packing the four files
of the path (gato/policy/{gato_policy,embeddings,input_tokenizers}.py, gato/transformers/trajectory_gpt2.py + the
package __init__ files), byte for byte, into ONE binary artefact: ``oracle/_ref/gato_ref.zip``, which oracle/ref_shim.py
unpacks into a scratch directory of the importing process.  No reference source file is placed in the tree.  oracle/_ref/ is git-ignored (never part of the
history) but not gpurun-ignored, so the archive travels to the box like the built .so; ``__graft_entry__.build()`` runs
this whenever /root/reference is present.  The in-memory shims of oracle/ref_shim.py are applied at import time as before."""
from __future__ import annotations

import hashlib
import os
import shutil
import sys
import zipfile

HERE = os.path.dirname(os.path.abspath(__file__))
DST = os.path.join(HERE, "_ref")
ARCHIVE = os.path.join(DST, "gato_ref.zip")
FILES = ["gato/__init__.py", "gato/policy/__init__.py", "gato/policy/gato_policy.py", "gato/policy/embeddings.py",
         "gato/policy/input_tokenizers.py", "gato/transformers/__init__.py", "gato/transformers/trajectory_gpt2.py"]


def build(src: str = "/root/reference", dst: str = DST) -> bool:
    """Returns True when <dst>/gato_ref.zip (by default oracle/_ref/gato_ref.zip) holds the reference's path files (packed now
    or already there)."""
    archive = os.path.join(dst, "gato_ref.zip")
    if not os.path.isfile(os.path.join(src, "gato", "policy", "gato_policy.py")):
        return os.path.isfile(archive)
    os.makedirs(dst, exist_ok=True)
    loose = os.path.join(dst, "gato")          # an earlier version of this recipe left loose files: remove them
    if os.path.isdir(loose):
        shutil.rmtree(loose)
    manifest = []
    tmp = archive + ".tmp"
    with zipfile.ZipFile(tmp, "w", compression=zipfile.ZIP_DEFLATED) as z:
        for rel in FILES:
            s = os.path.join(src, rel)
            data = open(s, "rb").read() if os.path.exists(s) else b""      # a package without an __init__.py in the reference
            info = zipfile.ZipInfo(rel, date_time=(2020, 1, 1, 0, 0, 0))   # fixed timestamps: reproducible archive
            info.compress_type = zipfile.ZIP_DEFLATED
            z.writestr(info, data)
            manifest.append(f"{hashlib.sha256(data).hexdigest()}  {rel}")
    os.replace(tmp, archive)
    with open(os.path.join(dst, "MANIFEST.sha256"), "w") as f:
        f.write("\n".join(manifest) + "\n")
    return True


if __name__ == "__main__":
    ok = build(sys.argv[1] if len(sys.argv) > 1 else "/root/reference")
    print("oracle/_ref:", "ready" if ok else "reference tree not found")
