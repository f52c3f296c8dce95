"""GPU parity against what the UNMODIFIED reference operator computes on a B200.

Reference side: hyvideo|hyvideo_i2v|wan/modules/attention_block_triton_diffres.py
`block_sparse_attention` — mask builder (ATen), `_triton_block_sparse_attn_fwd_kernel_onehot`
JIT-compiled by Triton for sm_100, text rows by FlashAttention-2 — run on a B200 on the inputs of
each case by tests/golden/make_reference_golden.py.  tests/golden/reference_parity.npz keeps a
seeded sample of its results: the mask rows of 32 image row blocks and the operator output at a
few hundred (token row, head) pairs.  Product side: the C-ABI library through
jenga_b200.attention, run here on the same inputs (the stored fingerprint proves they are).

What is asserted, in bf16 (the production dtype) and at BASELINE.json's shapes:

(1) attention kernel, given the REFERENCE'S mask rows (isolates a-9/a-10 from selection ties).
    Ground truth T = fp64 softmax attention of the same bf16 inputs on sampled query blocks.
    Measured on the B200 (profiles/r02_reference_parity.md): the reference's own Triton + FA2
    arithmetic deviates from T by max 1.6-1.9e-2*RMS, mean 2.2e-3*RMS (bf16); max 2.2e-3, mean
    2.6e-4 (fp16).  The stated tolerance follows from that, not from our kernel:
        err(product vs T) <= 1.5 * err(reference vs T)  (max)  and  <= 1.25 * (mean)
            — the product is no further from the exact result than the reference is;
        mean |product - reference| <= 2e-3 * RMS                 (SURVEY §8c-iv, unchanged)
        max  |product - reference| <= 3e-2 * RMS  (bf16), 5e-3 * RMS (fp16)
            — SURVEY §8c-iv wrote 2e-2 for the max; two implementations that are EACH up to
              1.9e-2 from T cannot be promised closer than ~2x that to each other (measured
              2.1-2.9e-2 between our kernel and the reference, 2.0e-2 between our dense class and
              FlashAttention-2, which itself sits 1.4e-2 from T), so the pairwise max bound is
              1.5x the survey's number and the error-vs-truth ratio carries the weight.
(2) selection (a-8) vs the reference builder on the GPU under torch.autocast(bf16): per-row counts
    equal on >= 98 % of rows, mean Jaccard >= 0.99 (SURVEY §8c-v), text columns exact.
(3) the whole operator (a-11): rows whose mask rows are identical obey the tolerance of (1); rows
    with different tie choices are a small fraction (<= 3 %).
Every statistic is taken over the stored sample.
"""
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
HERE = Path(__file__).resolve().parent
ROOT = HERE.parent
sys.path.insert(0, str(HERE))
sys.path.insert(0, str(ROOT))

import refutil  # noqa: E402

BLOCK = 128
GOLDEN = HERE / "golden" / "reference_parity.npz"


# name: (bench workload, heads used, dtype override)
CASES = {
    "hy_small": ("tiny", 2, None),
    "hy720p_3heads": ("hy720p", 3, None),
    "hy_turbo_s0_3heads": ("hy_turbo_s0", 3, None),
    "hy_i2v_3heads": ("hy_i2v", 3, None),
    "wan1.3b_full": ("wan1.3b", 12, None),
    "hy_small_fp16": ("tiny", 2, torch.float16),
}


def _inputs(case):
    import bench
    wl_name, heads, dt = CASES[case]
    wl = bench.workload(wl_name, 0.7)
    if wl_name == "tiny":
        wl = dict(wl, text_amp=0.431)
    dev = torch.device("cuda", 0)
    inp = bench.build_inputs(wl, dev, heads=heads, seed=4321)
    if dt is not None:
        for n in ("q", "k", "v"):
            inp[n] = inp[n].to(dt)
    return wl, inp


def _sample_blocks(n_img, text_blocks):
    img = sorted({0, 1, n_img // 3, n_img // 2, (2 * n_img) // 3, n_img - 2, n_img - 1} & set(range(n_img)))
    return img, [n_img + i for i in range(text_blocks)]


def fingerprint(inp):
    """sum|x| and sum x^2 of q, k, v in fp64: proves that the inputs are the ones the reference saw"""
    return np.array([f(inp[n].double()).item() for n in ("q", "k", "v")
                     for f in (lambda x: x.abs().sum(), lambda x: x.pow(2).sum())])


def _golden(case):
    with np.load(GOLDEN, allow_pickle=False) as z:
        g = {k.split("/", 1)[1]: z[k] for k in z.files if k.startswith(case + "/")}
    dt = getattr(torch, str(g["dtype"]))
    nb_bits = g["mask"].shape[-1] * 8
    g["mask"] = torch.from_numpy(np.unpackbits(g["mask"], axis=-1).astype(bool))
    g["out"] = torch.from_numpy(g["out"].view(np.int16)).view(dt)
    g["rows"] = torch.from_numpy(g["rows"]).long()
    g["heads"] = torch.from_numpy(g["heads"]).long()
    g["mask_blocks"] = torch.from_numpy(g["mask_blocks"]).long()
    g["nb_bits"] = nb_bits
    return g


def _at(x, S, H, rows, heads):
    """[1,S,H*128] or [1,S,H,128] -> [P,128]: the (token row, head) pairs of the sample."""
    return x.reshape(S, H, BLOCK)[rows.to(x.device), heads.to(x.device)]


@pytest.mark.parametrize("case", list(CASES))
def test_product_matches_unmodified_reference_operator(case):
    from jenga_b200.attention import (bits_to_onehot, block_sparse_attention_variant,
                                      carved_attention_fwd, mask_onehot_to_bits)
    g = _golden(case)
    wl, inp = _inputs(case)
    variant = wl["variant"]
    q, k, v, cu, nbr = inp["q"], inp["k"], inp["v"], inp["cu"], inp["nbr"]
    S, H = inp["S"], inp["heads"]
    nb = (S + BLOCK - 1) // BLOCK
    tb = wl["text_blocks"]
    n_img = nb - tb
    fp = fingerprint(inp)
    assert np.allclose(fp, g["fingerprint"], rtol=1e-9, atol=0), ("inputs differ from the stored case", fp, g["fingerprint"])
    dev = q.device
    mb = g["mask_blocks"].to(dev)
    ref_rows = g["mask"][..., :nb].to(dev)[None]                      # [1, H, len(mb), nb]
    assert ref_rows.shape == (1, H, len(mb), nb) and g["nb_bits"] - nb < 8
    rows, heads = g["rows"], g["heads"]
    ref_out = g["out"].to(dev)                                         # [P, 128]
    # ---------------- product: whole operator (own selection)
    out, bits = block_sparse_attention_variant(
        variant, q, k, v, inp["top_k"], cu_seqlens_q=cu, cu_seqlens_kv=cu, text_blocks=tb,
        text_amp=wl["text_amp"], block_neighbor_list=nbr, p_remain_rates=wl["p_remain"],
        first_frame_blocks=wl["first_frame"], return_mask_bits=True)
    torch.cuda.synchronize()
    assert out.dtype == ref_out.dtype and out.shape == (1, S, H * 128)
    got_mask = bits_to_onehot(bits, nb)
    same_rows, jac, counts, text_ok = refutil.mask_agreement(got_mask[:, :, mb], ref_rows, n_img)
    # ---------------- product kernel on the reference's mask rows (the other rows keep our own)
    mixed = got_mask.clone()
    mixed[:, :, mb] = ref_rows
    seqlen = int(cu[1].item()) if (cu is not None and variant != "wan") else S
    qb, kb, vb = (x if x.dtype in (torch.bfloat16, torch.float16) else x.to(torch.bfloat16) for x in (q, k, v))
    attn = carved_attention_fwd(
        qb, kb, vb, mask_onehot_to_bits(mixed), nq_sparse=n_img, nq_dense=tb, sm_scale=128 ** -0.5,
        text_amp=wl["text_amp"], text_block_start=n_img, kv_limit_sparse=seqlen, q_limit_sparse=seqlen,
        kv_limit_dense=nb * BLOCK)
    torch.cuda.synchronize()
    attn_p = _at(attn.to(ref_out.dtype), S, H, rows, heads)
    out_p = _at(out, S, H, rows, heads)
    blk = rows // BLOCK
    is_txt = (blk >= n_img).to(dev)
    # ---------------- fp64 ground truth on sampled blocks
    img_blocks, txt_blocks = _sample_blocks(n_img, tb)
    truth = refutil.fp64_truth(qb, kb, vb, mixed, img_blocks + txt_blocks, n_img_blocks=n_img,
                               seqlen=seqlen, text_amp=wl["text_amp"])
    stats = {}
    for tag, tblocks in (("img", img_blocks), ("txt", txt_blocks)):
        sel = torch.tensor([int(b) in tblocks for b in blk], dtype=torch.bool)
        if not sel.any():
            continue
        t = torch.stack([truth[int(r) // BLOCK][int(h), int(r) % BLOCK] for r, h in zip(rows[sel], heads[sel])])
        rms = t.pow(2).mean().sqrt().item() + 1e-30
        r_err = (ref_out[sel.to(dev)].double() - t).abs()
        p_err = (attn_p[sel.to(dev)].double() - t).abs()
        stats[tag] = dict(ref_max=r_err.max().item() / rms, ref_mean=r_err.mean().item() / rms,
                          prod_max=p_err.max().item() / rms, prod_mean=p_err.mean().item() / rms, rms=rms)
    # product vs reference on the sampled pairs
    d_max, d_mean = refutil.pair_stats(attn_p[~is_txt], ref_out[~is_txt])
    d_txt = refutil.pair_stats(attn_p[is_txt], ref_out[is_txt]) if tb else (0.0, 0.0)
    # whole operator: sampled image pairs whose mask rows are identical to the reference's
    row_same = (got_mask[:, :, mb] == ref_rows).all(-1)[0]           # [H, len(mb)]
    pos = torch.full((n_img,), -1, dtype=torch.long, device=dev)
    pos[mb] = torch.arange(len(mb), device=dev)
    img_idx = (~is_txt).nonzero()[:, 0]
    sel = row_same[heads.to(dev)[img_idx], pos[blk.to(dev)[img_idx]]]
    diff = (out_p[img_idx].float() - ref_out[img_idx].float()).abs()
    rms_all = ref_out[img_idx].float().pow(2).mean().sqrt().item()
    op_max = (diff * sel[:, None]).max().item() / rms_all
    op_mean = ((diff * sel[:, None]).sum() / (sel.sum() * 128).clamp_min(1)).item() / rms_all
    rec = dict(case=case, dtype=str(qb.dtype), S=S, heads=H, pairs=len(rows),
               mask_same_rows=same_rows, mask_jaccard=jac, mask_counts_equal=counts,
               kernel_vs_ref_max=d_max, kernel_vs_ref_mean=d_mean, text_vs_fa2_max=d_txt[0],
               text_vs_fa2_mean=d_txt[1], operator_vs_ref_max=op_max, operator_vs_ref_mean=op_mean, **{
                   f"{t}_{n}": val for t, s_ in stats.items() for n, val in s_.items()})
    print("\n[reference parity]", rec)

    fp16 = qb.dtype == torch.float16
    a_max, a_mean = (5e-3, 5e-4) if fp16 else (3e-2, 2e-3)
    # (2) selection
    assert text_ok
    assert counts >= 0.98 and jac >= 0.99, (counts, jac)
    assert same_rows >= 0.97, same_rows
    # (1) kernel on the reference's mask
    assert d_max <= a_max and d_mean <= a_mean, ("sparse rows vs reference Triton kernel", d_max, d_mean)
    assert d_txt[0] <= a_max and d_txt[1] <= a_mean, ("text rows vs FlashAttention-2", d_txt)
    for tag, s_ in stats.items():
        assert s_["prod_max"] <= 1.5 * s_["ref_max"] + 1e-4, (tag, s_)
        assert s_["prod_mean"] <= 1.25 * s_["ref_mean"] + 1e-5, (tag, s_)
    # (3) operator
    assert op_max <= a_max and op_mean <= a_mean, (op_max, op_mean)
    # rows at or past seqlen of the image part are zeros, as in the reference (…:136,:156)
    if seqlen < n_img * BLOCK:
        assert (out.reshape(1, S, H, 128)[0, seqlen:n_img * BLOCK] == 0).all()


def test_dense_shims_match_installed_flash_attn():
    """a-10 / the FlashAttention call sites (SURVEY §8b): our flash_attn_func / flash_attn_varlen_func
    shims against the INSTALLED flash_attn wheel (third-party, the reference's own dependency) in
    bf16, judged against fp64 truth like (1)."""
    flash_attn = pytest.importorskip("flash_attn")
    from flash_attn.flash_attn_interface import flash_attn_varlen_func as fa_varlen
    from jenga_b200 import flash_attn_shim as F
    g = torch.Generator(device="cuda").manual_seed(99)
    B, S, H, D = 1, 128 * 37 + 56, 4, 128
    q, k, v = (torch.randn(B, S, H, D, generator=g, device="cuda").bfloat16() for _ in range(3))
    ref = flash_attn.flash_attn_func(q, k, v, causal=False, softmax_scale=D ** -0.5)
    got = F.flash_attn_func(q, k, v, causal=False, softmax_scale=D ** -0.5)
    nb = (S + 127) // 128
    ones = torch.ones(1, H, 0, nb, dtype=torch.bool, device="cuda")
    truth = refutil.fp64_truth(q, k, v, ones, [0, nb // 2, nb - 1], n_img_blocks=0, seqlen=S)
    # the shim's dense class sees exactly S keys; truth pads with zero keys -> restrict by masking:
    # recompute truth without padding influence
    kd, vd = k[0].transpose(0, 1).double(), v[0].transpose(0, 1).double()
    truth = {}
    for qb in (0, nb // 2, nb - 1):
        Q = q[0, qb * 128:(qb + 1) * 128].transpose(0, 1).double()
        p = torch.softmax(torch.matmul(Q, kd.transpose(1, 2)) * D ** -0.5, dim=-1)
        t = torch.matmul(p, vd)
        if t.shape[1] < 128:
            t = torch.nn.functional.pad(t, [0, 0, 0, 128 - t.shape[1]])
        truth[qb] = t
    r_max, r_mean, _ = refutil.error_stats(ref, truth)
    p_max, p_mean, _ = refutil.error_stats(got, truth)
    d_max, d_mean = refutil.pair_stats(got, ref)
    print(f"\n[fa2 parity] dense: ours-vs-fa2 max {d_max:.2e} mean {d_mean:.2e}; vs fp64: fa2 {r_max:.2e}/{r_mean:.2e} "
          f"ours {p_max:.2e}/{p_mean:.2e}")
    assert d_max <= 3e-2 and d_mean <= 2e-3
    assert p_max <= 1.5 * r_max + 1e-4 and p_mean <= 1.25 * r_mean + 1e-5
    # varlen form used by hyvideo/modules/attenion.py:109-117: two segments [0,s1) and [s1,S)
    s1 = 128 * 20 + 17
    cu = torch.tensor([0, s1, S], dtype=torch.int32, device="cuda")
    qf, kf, vf = (x.reshape(S, H, D) for x in (q, k, v))
    ref_v = fa_varlen(qf, kf, vf, cu, cu, S, S)
    got_v = F.flash_attn_varlen_func(qf, kf, vf, cu, cu, S, S)
    dv_max, dv_mean = refutil.pair_stats(got_v, ref_v)
    print(f"[fa2 parity] varlen: max {dv_max:.2e} mean {dv_mean:.2e}")
    assert dv_max <= 3e-2 and dv_mean <= 2e-3


def test_flash_attn_forward_shim_returns_lse_like_installed_flash_attn():
    """flash_attn.flash_attn_interface._flash_attn_forward (hyvideo/modules/attenion.py:221-246,
    xdit_ring_atten.py:302-327): (out, softmax_lse, ...) — out as above, lse within 2e-3 absolute of
    the installed wheel's (fp32 natural-log LSE; ours comes from a base-2 running max + sum)."""
    pytest.importorskip("flash_attn")
    from flash_attn.flash_attn_interface import _flash_attn_forward as fa_fwd
    from jenga_b200 import flash_attn_shim as F
    g = torch.Generator(device="cuda").manual_seed(7)
    B, Sq, Sk, H, D = 1, 300, 128 * 9 + 40, 3, 128
    q = torch.randn(B, Sq, H, D, generator=g, device="cuda").bfloat16()
    k = torch.randn(B, Sk, H, D, generator=g, device="cuda").bfloat16()
    v = torch.randn(B, Sk, H, D, generator=g, device="cuda").bfloat16()
    ref = fa_fwd(q, k, v, dropout_p=0.0, softmax_scale=D ** -0.5, causal=False, window_size_left=-1,
                 window_size_right=-1, softcap=0.0, alibi_slopes=None, return_softmax=False)
    got = F._flash_attn_forward(q, k, v, dropout_p=0.0, softmax_scale=D ** -0.5, causal=False, window_size_left=-1,
                                window_size_right=-1, softcap=0.0, alibi_slopes=None, return_softmax=False)
    ro, rl = ref[0], ref[1]
    go, gl = got[0], got[1]
    assert gl.shape == rl.shape == (B, H, Sq) and gl.dtype == torch.float32
    truth = torch.logsumexp(torch.einsum("bqhd,bkhd->bhqk", q.double(), k.double()) * D ** -0.5, dim=-1)
    print(f"\n[fa2 lse] |ours-fa2| max {(gl - rl).abs().max().item():.2e}; vs fp64: fa2 {(rl - truth).abs().max().item():.2e} "
          f"ours {(gl - truth).abs().max().item():.2e}")
    assert (gl.double() - truth).abs().max().item() <= 2e-3
    assert (gl - rl).abs().max().item() <= 2e-3
    d_max, d_mean = refutil.pair_stats(go, ro)
    assert d_max <= 3e-2 and d_mean <= 2e-3

