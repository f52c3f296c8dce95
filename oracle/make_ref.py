#!/usr/bin/env python
"""TEST INFRASTRUCTURE — materialises oracle/_ref/: the UNMODIFIED reference files of the hot path.

The reference (dvlab-research/Jenga) is pure Python + one Triton kernel; "building" it means
putting the handful of files SURVEY §8(a) cites where the GPU box can import them.  This recipe
copies them byte for byte from /root/reference (read-only, present only in the build container)
into oracle/_ref/ (git-ignored: never in history; NOT gpurun-ignored: it travels with the
snapshot like our own built .so) and writes MANIFEST.json with their SHA-256.  Nothing is edited.

Run by __graft_entry__.build() and `make -C oracle ref`.  On the GPU box /root/reference does
not exist; oracle/ref_loader.py then imports from oracle/_ref/ only.

Consumers (checker only — never the product): tests/test_reference_gpu.py,
tests/test_install_reference_*.py, bench.py's `gpu_reference` leg.
"""
from __future__ import annotations

import hashlib
import json
import os
import shutil
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
DST = HERE / "_ref"
SRC = Path("/root/reference")

# every file is on the hot path (SURVEY §8a) or is imported by one that is
FILES = [
    "gilbert.py",
    "jenga_hyvideo.py", "jenga_hyvideo_multigpu.py", "jenga_hyi2v.py", "jenga_wan.py",
    "hyvideo/modules/attention_block_triton_diffres.py",
    "hyvideo/modules/norm_layers.py",
    "hyvideo/modules/posemb_layers.py",
    "hyvideo/modules/attenion.py",
    "hyvideo/modules/activation_layers.py",
    "hyvideo/modules/embed_layers.py",
    "hyvideo/modules/mlp_layers.py",
    "hyvideo/modules/modulate_layers.py",
    "hyvideo/modules/token_refiner.py",
    "hyvideo/modules/models_mul_block_gc_ha_multigpu.py",
    "hyvideo/modules/xdit_ring_atten.py",
    "hyvideo/utils/helpers.py",
    "hyvideo_i2v/modules/attention_block_triton_diffres.py",
    "hyvideo_i2v/modules/norm_layers.py",
    "hyvideo_i2v/modules/posemb_layers.py",
    "hyvideo_i2v/modules/attenion.py",
    "hyvideo_i2v/modules/activation_layers.py",
    "hyvideo_i2v/modules/embed_layers.py",
    "hyvideo_i2v/modules/mlp_layers.py",
    "hyvideo_i2v/modules/modulate_layers.py",
    "hyvideo_i2v/modules/token_refiner.py",
    "hyvideo_i2v/modules/models_mul.py",
    "hyvideo_i2v/utils/helpers.py",
    "wan/modules/attention_block_triton_diffres.py",
    "wan/modules/attention.py",
    "wan/modules/model_mul.py",
]


def readable_dir(p: Path) -> bool:
    """True iff `p` is a directory this process may read (a directory behind one it may not
    enter counts as absent instead of raising PermissionError)."""
    try:
        return p.is_dir() and os.access(p, os.R_OK | os.X_OK)
    except OSError:
        return False


def materialise(src: Path = SRC, dst: Path = DST, quiet: bool = False) -> Path | None:
    """Copies FILES from `src` to `dst`.  Returns dst, or None when the reference is not mounted
    and nothing was materialised earlier (callers skip reference-backed checks then)."""
    if not readable_dir(src):
        return dst if (dst / "MANIFEST.json").exists() else None
    manifest = {}
    for rel in FILES:
        s = src / rel
        if not s.is_file():
            continue
        d = dst / rel
        d.parent.mkdir(parents=True, exist_ok=True)
        data = s.read_bytes()
        if not d.exists() or d.read_bytes() != data:
            shutil.copyfile(s, d)
        manifest[rel] = hashlib.sha256(data).hexdigest()
    (dst / "MANIFEST.json").write_text(json.dumps(
        {"source": str(src), "note": "byte-for-byte copies, see oracle/make_ref.py", "files": manifest},
        indent=1, sort_keys=True))
    if not quiet:
        print(f"[make_ref] {len(manifest)} reference files -> {dst}")
    return dst


def verify(dst: Path = DST) -> bool:
    """True iff every file under dst still hashes to its manifest entry (i.e. is unmodified)."""
    mf = dst / "MANIFEST.json"
    if not mf.exists():
        return False
    files = json.loads(mf.read_text())["files"]
    return all((dst / rel).is_file() and hashlib.sha256((dst / rel).read_bytes()).hexdigest() == h
               for rel, h in files.items())


if __name__ == "__main__":
    out = materialise()
    if out is None:
        print("[make_ref] /root/reference not mounted and no earlier oracle/_ref/ — nothing to do")
        sys.exit(0)
    assert verify(out)
