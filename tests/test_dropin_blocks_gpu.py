"""The drop-in, proven on REAL reference code: the unmodified block classes of
hyvideo/modules/models_mul_block_gc_ha_multigpu.py (MMDoubleStreamBlock :43-316,
MMSingleStreamBlock :319-500) and wan/modules/model_mul.py (WanSelfAttention :105-180) are imported
twice from the reference tree (oracle/ref_loader.py) —

  A: bound to the reference's own operator (Triton JIT + FlashAttention-2),
  B: through jenga_b200.install.install(): operator modules pre-seeded, block forwards patched by
     the import hook so RMSNorm + RoPE + cat + pooling run as the fused prologue kernel, token
     reorders routed to the gather kernel —

given the SAME random-init weights and inputs on the GPU, and compared.  Tolerance: rows whose
selection masks are identical in every head (>= 90 % of rows; the rest differ only by the
reference's unstable tie order) obey |B - A| <= 3e-2*RMS + 2^-7*|A| per element and 3e-3*RMS mean on
the block OUTPUT (the attention tolerance of test_reference_gpu.py propagated through proj + MLP +
residual, plus one bf16 ulp of the output)."""
import sys
from pathlib import Path

import pytest
import torch

pytestmark = pytest.mark.gpu
HERE = Path(__file__).resolve().parent
ROOT = HERE.parent
sys.path.insert(0, str(HERE))
sys.path.insert(0, str(ROOT))


@pytest.fixture(scope="module")
def modules():
    from oracle import ref_loader as R
    if not R.available():
        pytest.skip("reference files not staged (oracle/_ref/)")
    ref_hy, ref_wan = R.load_blocks(product=False)
    our_hy, our_wan = R.load_blocks(product=True)
    assert not getattr(ref_hy.MMDoubleStreamBlock.forward, "__jenga_b200__", False)
    assert our_hy.MMDoubleStreamBlock.forward.__jenga_b200__
    assert our_hy.block_sparse_attention.__doc__.startswith("jenga_b200 drop-in")
    assert "_triton_block_sparse_attention_onehot" in ref_hy.block_sparse_attention.__globals__
    yield ref_hy, ref_wan, our_hy, our_wan
    from jenga_b200 import blocks
    blocks.remove_gather_hook()


def _reinit(module, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    with torch.no_grad():
        for n, p in module.named_parameters():
            if p.dim() >= 2:
                p.copy_(torch.randn(p.shape, generator=g, device="cuda") * (0.6 / p.shape[-1] ** 0.5))
            elif "norm" in n and n.endswith("weight"):
                p.copy_(1.0 + 0.2 * torch.randn(p.shape, generator=g, device="cuda"))
            else:
                p.copy_(0.05 * torch.randn(p.shape, generator=g, device="cuda"))


def _structured_tokens(L, C, seed, gain=3.0):
    """hidden states with per-128-token-block structure so that block scores are well separated"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    nb = L // 128
    c = torch.randn(nb, C, generator=g, device="cuda")
    c = torch.nn.functional.avg_pool1d(torch.nn.functional.pad(c.t()[None], (1, 1), mode="replicate"), 3, 1)[0].t()
    x = torch.randn(L, C, generator=g, device="cuda") + gain * c.repeat_interleave(128, 0)
    return x[None].to(torch.bfloat16)


def _capture_reference_masks(ref_operator_fn):
    """Wraps (does not edit) the reference builder inside the module `ref_operator_fn` lives in."""
    g = ref_operator_fn.__globals__
    rec = []
    orig = g["_build_block_index_with_importance_optimized"]

    def wrapped(*a, **k):
        m = orig(*a, **k)
        rec.append(m)
        return m
    g["_build_block_index_with_importance_optimized"] = wrapped
    return rec, lambda: g.__setitem__("_build_block_index_with_importance_optimized", orig)


def _rows_with_equal_masks(ref_mask, our_bits, nb):
    from jenga_b200.attention import bits_to_onehot
    ours = bits_to_onehot(our_bits, nb)
    same = (ours == ref_mask).all(-1).all(1)[0]      # [n_img blocks]: equal in every head
    return same


def _compare(a, b, row_ok, what):
    """per element |B - A| <= 3e-2*RMS + 2^-7*|A| (the |A| term admits one bf16 ulp flip of the
    block output, which carries the residual stream), mean <= 3e-3*RMS, on rows with equal masks"""
    a, b = a.float(), b.float()
    rms = a.pow(2).mean().sqrt().item()
    d = (a - b).abs()[0]                              # [rows, C]
    sel = row_ok[:, None]
    frac = row_ok.float().mean().item()
    bad = ((d > 3e-2 * rms + 2.0 ** -7 * a.abs()[0]) & sel).sum().item()
    mx = (d * sel).max().item() / rms
    mean = ((d * sel).sum() / (sel.sum() * d.shape[1]).clamp_min(1)).item() / rms
    print(f"\n[drop-in] {what}: rows with identical masks {frac:.3f}, max {mx:.3e} mean {mean:.3e} (x RMS), "
          f"{bad} elements over the bound")
    assert frac >= 0.90, (what, frac)
    assert bad == 0 and mean <= 3e-3, (what, mx, mean, bad)


def _hy_case(hy_mod):
    from jenga_b200 import gilbert
    t, h, w = 8, 16, 16
    L, T, C, H = t * h * w, 256, 512, 4
    l2h, h2l = gilbert.mapping_tensors(t, h, w)
    nbr = gilbert.block_neighbor_mapping(t, h, w)
    curve_sel = [[l2h.cuda(), h2l.cuda(), nbr]]
    img = _structured_tokens(L, C, 1)
    txt = _structured_tokens(T, C, 2, gain=0.5)
    vec = torch.randn(1, C, generator=torch.Generator(device="cuda").manual_seed(3), device="cuda").bfloat16()
    text_mask = torch.zeros(1, T, dtype=torch.int64, device="cuda")
    text_mask[:, :180] = 1
    cu = hy_mod.get_cu_seqlens(text_mask, L)
    ang = torch.rand(L, 64, generator=torch.Generator(device="cuda").manual_seed(4), device="cuda") * 6.2831853
    freqs = (torch.cos(ang).repeat_interleave(2, dim=1).contiguous(), torch.sin(ang).repeat_interleave(2, dim=1).contiguous())
    return dict(L=L, T=T, C=C, H=H, curve_sel=curve_sel, img=img, txt=txt, vec=vec, cu=cu, freqs=freqs)


@pytest.mark.parametrize("kind", ["double", "single"])
def test_unmodified_hunyuan_blocks_through_install_hook(modules, kind):
    ref_hy, _, our_hy, _ = modules
    from jenga_b200 import attention as A, blocks
    c = _hy_case(ref_hy)
    cls = "MMDoubleStreamBlock" if kind == "double" else "MMSingleStreamBlock"
    mk = lambda m: getattr(m, cls)(c["C"], c["H"], mlp_width_ratio=4.0, dtype=torch.bfloat16, device="cuda")  # noqa: E731
    ref_blk, our_blk = mk(ref_hy), mk(our_hy)
    _reinit(ref_blk, 11)
    our_blk.load_state_dict(ref_blk.state_dict())
    kw = dict(sa_drop_rate=0.7, txt_amp=0.431, curve_sel=c["curve_sel"], p_remain_rates=0.3)
    rec, undo = _capture_reference_masks(ref_hy.block_sparse_attention)
    before = dict(blocks.STATS)
    A.MASK_CAPTURE = []
    try:
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            if kind == "double":
                ra = ref_blk(c["img"], c["txt"], c["vec"], c["cu"], c["cu"], c["L"] + c["T"], c["L"] + c["T"], c["freqs"], **kw)
                oa = our_blk(c["img"], c["txt"], c["vec"], c["cu"], c["cu"], c["L"] + c["T"], c["L"] + c["T"], c["freqs"], **kw)
            else:
                x = torch.cat([c["img"], c["txt"]], 1)
                ra = (ref_blk(x, c["vec"], c["T"], c["cu"], c["cu"], c["L"] + c["T"], c["L"] + c["T"], c["freqs"], **kw),)
                oa = (our_blk(x, c["vec"], c["T"], c["cu"], c["cu"], c["L"] + c["T"], c["L"] + c["T"], c["freqs"], **kw),)
        torch.cuda.synchronize()
        bits, nb = A.MASK_CAPTURE[-1]
    finally:
        A.MASK_CAPTURE = None
        undo()
    key = "hy_double" if kind == "double" else "hy_single"
    assert blocks.STATS[key] == before[key] + 1, "the fused attention section did not run"
    assert len(rec) == 1
    same_blocks = _rows_with_equal_masks(rec[0], bits, nb)
    row_ok = same_blocks.repeat_interleave(128)
    _compare(ra[0][:, :c["L"]], oa[0][:, :c["L"]], row_ok, f"{cls} image rows")
    txt_a = ra[1] if kind == "double" else ra[0][:, c["L"]:]
    txt_b = oa[1] if kind == "double" else oa[0][:, c["L"]:]
    _compare(txt_a, txt_b, torch.ones(c["T"], dtype=torch.bool, device="cuda"), f"{cls} text rows")


def test_unmodified_wan_self_attention_through_install_hook(modules):
    _, ref_wan, _, our_wan = modules
    from jenga_b200 import attention as A, blocks, gilbert
    f, h, w = 21, 12, 16                     # 4032 tokens -> 32 blocks (ragged: 4032 = 31.5 blocks)
    L, dim, H = f * h * w, 512, 4
    l2h, h2l = gilbert.mapping_tensors(f, h, w, sliced=True)
    nbr = gilbert.block_neighbor_mapping(f, h, w, sliced=True)
    mk = lambda m: m.WanSelfAttention(dim, H).cuda()   # noqa: E731
    ref_sa, our_sa = mk(ref_wan), mk(our_wan)
    _reinit(ref_sa, 21)
    our_sa.load_state_dict(ref_sa.state_dict())
    x = _structured_tokens(L - L % 128, dim, 5)
    x = torch.cat([x, _structured_tokens(128, dim, 6)[:, : L % 128]], 1).float()
    d = dim // H
    freqs = torch.cat([ref_wan.rope_params(1024, d - 4 * (d // 6)), ref_wan.rope_params(1024, 2 * (d // 6)),
                       ref_wan.rope_params(1024, 2 * (d // 6))], dim=1).cuda()
    grid = torch.tensor([[f, h, w]])
    seq_lens = torch.tensor([L])
    kw = dict(sa_drop_rate=0.5, p_remain_rates=0.9, freq_remap=h2l.cuda(), block_neighbor_list=nbr)
    rec, undo = _capture_reference_masks(ref_wan.block_sparse_attention)
    before = dict(blocks.STATS)
    A.MASK_CAPTURE = []
    try:
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            ra = ref_sa(x, seq_lens, grid, freqs, **kw)
            oa = our_sa(x, seq_lens, grid, freqs, **kw)
        torch.cuda.synchronize()
        bits, nb = A.MASK_CAPTURE[-1]
    finally:
        A.MASK_CAPTURE = None
        undo()
    assert blocks.STATS["wan_self"] == before["wan_self"] + 1
    assert ra.dtype == oa.dtype and ra.shape == oa.shape
    same_blocks = _rows_with_equal_masks(rec[0], bits, nb)
    row_ok = same_blocks.repeat_interleave(128)[:L]
    _compare(ra, oa, row_ok, "WanSelfAttention")


def test_token_reorder_is_routed_to_the_gather_kernel():
    """jenga_hyvideo.py:116-118,226: img[:, hilbert_order], freqs[hilbert_order], img[:, linear_to_hilbert].
    Needs no reference file: the hook sees plain tensor indexing."""
    from jenga_b200 import blocks, gilbert
    l2h, h2l = gilbert.mapping_tensors(8, 16, 16)
    l2h, h2l = l2h.cuda(), h2l.cuda()
    img = torch.randn(1, 2048, 512, device="cuda").bfloat16()
    cos = torch.randn(2048, 128, device="cuda")
    was_installed = blocks._gather_mode is not None
    blocks.install_gather_hook()
    before = blocks.STATS["gather"]
    a = img[:, h2l]
    b = cos[h2l]
    back = a[:, l2h]
    assert blocks.STATS["gather"] == before + 3
    blocks.remove_gather_hook()
    try:
        assert torch.equal(a, img[:, h2l]) and torch.equal(b, cos[h2l]) and torch.equal(back, img)
    finally:
        if was_installed:
            blocks.install_gather_hook()
