"""TEST INFRASTRUCTURE — imports the UNMODIFIED reference files (checker only, never the product).

Where the reference lives: /root/reference in the build container, oracle/_ref/ (materialised by
oracle/make_ref.py, byte-for-byte copies, SHA manifest) on the GPU box.  Nothing here edits a
reference file; what it supplies is the *environment* the files expect and this image lacks:

* `matplotlib*`                — gilbert.py's plotting imports (gilbert.py:1-10), never called.
* `diffusers` mixins           — base classes of the DiT classes; the block classes
                                  (MMDoubleStreamBlock, MMSingleStreamBlock, WanSelfAttention)
                                  are plain nn.Modules and do not use them.
* `xfuser.core.distributed`    — sequence-parallel world size / rank queries
                                  (models_mul_block_gc_ha_multigpu.py:26-30); answered from
                                  torch.distributed (1 / 0 when not initialised).
* synthetic `hyvideo`, `hyvideo.modules`, `hyvideo.utils`, `hyvideo_i2v…`, `wan`, `wan.modules`
  packages whose __path__ points into the reference tree, so that the packages' own
  __init__.py (which import the whole pipeline: diffusers, transformers checkpoints, …) are
  not executed but relative imports between the hot-path files resolve normally.

Only tests/, __graft_entry__.smoke() and bench.py's reference legs import this module.
"""
from __future__ import annotations

import contextlib
import importlib
import importlib.util
import sys
import types
from pathlib import Path

HERE = Path(__file__).resolve().parent
_PKGS = ("hyvideo", "hyvideo_i2v", "wan")


def ref_root() -> Path | None:
    """The directory holding the unmodified reference files, or None."""
    import os
    live = Path("/root/reference")
    from . import make_ref
    if make_ref.readable_dir(live) and (live / "gilbert.py").is_file() and os.environ.get("JENGA_ORACLE_REF") != "staged":
        return live
    staged = HERE / "_ref"
    if (staged / "MANIFEST.json").is_file():
        if not make_ref.verify(staged):
            raise RuntimeError("oracle/_ref/ does not match its manifest: the reference copy was modified")
        return staged
    return None


def available() -> bool:
    return ref_root() is not None


def _stub(name: str, **attrs) -> types.ModuleType:
    m = sys.modules.get(name)
    if m is None:
        m = types.ModuleType(name)
        m.__dict__["__oracle_stub__"] = True
        sys.modules[name] = m
    for k, v in attrs.items():
        if not hasattr(m, k):
            setattr(m, k, v)
    return m


def install_environment_stubs() -> None:
    """Stubs for the third-party packages the reference imports and this image lacks."""
    import torch

    for n in ("matplotlib", "matplotlib.pyplot", "mpl_toolkits", "mpl_toolkits.mplot3d"):
        try:
            importlib.import_module(n)
        except Exception:
            _stub(n, Axes3D=object)
    try:
        import diffusers  # noqa: F401
    except Exception:
        _stub("diffusers")
        _stub("diffusers.configuration_utils", ConfigMixin=object, register_to_config=lambda f: f)
        _stub("diffusers.models", ModelMixin=torch.nn.Module)
        _stub("diffusers.models.modeling_utils", ModelMixin=torch.nn.Module)
    try:
        import xfuser.core.distributed  # noqa: F401
    except Exception:
        import torch.distributed as dist

        def _ws():
            return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1

        def _rk():
            return dist.get_rank() if dist.is_available() and dist.is_initialized() else 0

        class _Group:
            world_size = property(lambda self: _ws())

            def all_gather(self, x, dim=0):
                if _ws() == 1:
                    return x
                outs = [torch.empty_like(x) for _ in range(_ws())]
                dist.all_gather(outs, x.contiguous())
                return torch.cat(outs, dim=dim)

        _stub("xfuser")
        _stub("xfuser.core")
        _stub("xfuser.core.distributed", get_sequence_parallel_world_size=_ws,
              get_sequence_parallel_rank=_rk, get_sp_group=lambda: _Group())


def import_by_path(name: str, rel: str):
    """Imports one standalone reference file (no relative imports) under a private module name."""
    root = ref_root()
    if root is None:
        raise FileNotFoundError("reference not available (neither /root/reference nor oracle/_ref/)")
    install_environment_stubs()
    if name in sys.modules:
        return sys.modules[name]
    spec = importlib.util.spec_from_file_location(name, root / rel)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    try:
        spec.loader.exec_module(mod)
    except Exception:
        sys.modules.pop(name, None)
        raise
    return mod


def operator(variant: str):
    """The reference's attention_block_triton_diffres module of one variant
    (hyvideo | hyvideo_i2v | wan), imported under a private name."""
    assert variant in _PKGS
    return import_by_path(f"_jenga_ref_op_{variant}", f"{variant}/modules/attention_block_triton_diffres.py")


def gilbert():
    return import_by_path("_jenga_ref_gilbert", "gilbert.py")


def _purge_packages() -> dict:
    saved = {}
    for k in list(sys.modules):
        if k.split(".")[0] in _PKGS:
            saved[k] = sys.modules.pop(k)
    return saved


@contextlib.contextmanager
def reference_packages(product: bool = False):
    """Context in which `import hyvideo.modules.<file>` / `import wan.modules.<file>` resolve to the
    unmodified reference files.  product=False: the files see the reference's own Triton/FA2
    operator.  product=True: jenga_b200.install.install() has pre-seeded sys.modules first, so the
    same unmodified files bind the B200 path at import time (the drop-in under test).
    Module objects imported inside stay usable after exit; sys.modules is restored so that a
    second context can import the same files with the other binding."""
    root = ref_root()
    if root is None:
        raise FileNotFoundError("reference not available")
    install_environment_stubs()
    saved = _purge_packages()
    saved_extra = {k: sys.modules.get(k) for k in ("flash_attn", "flash_attn.flash_attn_interface", "gilbert")}
    # a pure-reference import must not be touched by the product's block-forward hook
    parked = [f for f in sys.meta_path if type(f).__name__ == "_PatchFinder"] if not product else []
    for f in parked:
        sys.meta_path.remove(f)
    try:
        if product:
            from jenga_b200 import install as _inst
            _inst.install()
        for pkg in _PKGS:
            for sub in ("", ".modules", ".utils"):
                name = pkg + sub
                if name in sys.modules:
                    continue
                m = types.ModuleType(name)
                m.__path__ = [str(root / name.replace(".", "/"))]
                m.__dict__["__oracle_stub__"] = True
                sys.modules[name] = m
        yield root
    finally:
        for f in parked:
            sys.meta_path.insert(0, f)
        _purge_packages()
        sys.modules.update(saved)
        for k, v in saved_extra.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def load_blocks(product: bool):
    """(hy_blocks_module, wan_model_module) = the unmodified
    hyvideo/modules/models_mul_block_gc_ha_multigpu.py and wan/modules/model_mul.py, bound to the
    reference operator (product=False) or to jenga_b200 through install() (product=True)."""
    with reference_packages(product=product):
        hy = importlib.import_module("hyvideo.modules.models_mul_block_gc_ha_multigpu")
        wan = importlib.import_module("wan.modules.model_mul")
    return hy, wan
