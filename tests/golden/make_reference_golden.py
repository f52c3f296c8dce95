#!/usr/bin/env python
"""Generates tests/golden/reference_parity.npz: what the UNMODIFIED reference operator computes on
a GPU for the cases of tests/test_reference_gpu.py, sampled small enough to commit.

Needs a CUDA device and the original project's files reachable through oracle/ref_loader.py
(its Triton kernel and FlashAttention-2 run as they are):

    python tests/golden/make_reference_golden.py [OUT.npz]

Per case `c` the file holds
    c/fingerprint   sum|x| and sum x^2 of q, k, v in fp64 (the inputs the reference saw)
    c/mask_blocks   image row blocks whose reference mask rows are stored
    c/mask          those rows, [H, len(mask_blocks), nb] bool packed along the last axis
    c/rows, c/heads (token row, head) pairs at which the reference output is stored
    c/out           the reference output at those pairs, [P, 128] values of c/dtype kept bit for
                    bit as 16-bit words (numpy has no bfloat16)
    c/dtype         "bfloat16", "float16" or "float32" (the wan variant returns float32)
The pairs are a seeded sample: every query block the fp64 ground truth of the test uses gets
TRUTH_PAIRS pairs, every other stored mask block OTHER_PAIRS, every text block TEXT_PAIRS.
"""
import sys
from pathlib import Path

import numpy as np
import torch

HERE = Path(__file__).resolve().parent
TESTS = HERE.parent
sys.path.insert(0, str(TESTS))
sys.path.insert(0, str(TESTS.parent))

import refutil  # noqa: E402
import test_reference_gpu as T  # noqa: E402

MASK_BLOCKS = 32
TRUTH_PAIRS, OTHER_PAIRS, TEXT_PAIRS = 10, 2, 12


def _pairs(rng, blk, n, row_end, heads):
    lo, hi = blk * 128, min(blk * 128 + 128, row_end)
    if hi <= lo:
        return []
    rows = rng.integers(lo, hi, size=n)
    return [(int(r), int(h)) for r, h in zip(rows, rng.integers(0, heads, size=n))]


def case_golden(case, seed):
    from oracle import ref_loader
    wl, inp = T._inputs(case)
    variant = wl["variant"]
    op = ref_loader.operator(variant)
    q, k, v, cu, nbr = inp["q"], inp["k"], inp["v"], inp["cu"], inp["nbr"]
    S, H = inp["S"], inp["heads"]
    nb = (S + 127) // 128
    tb = wl["text_blocks"]
    n_img = nb - tb
    kw = dict(top_k=inp["top_k"], text_blocks=tb, nbr=nbr, p_remain=wl["p_remain"], first_frame=wl["first_frame"])
    ref_mask = refutil.reference_mask(op, variant, q, k, **kw)
    assert torch.equal(ref_mask, refutil.reference_mask(op, variant, q, k, **kw)), "reference builder not deterministic"
    ref_out = refutil.reference_call(op, variant, q, k, v, cu=cu, text_amp=wl["text_amp"], **kw)
    torch.cuda.synchronize()
    assert ref_out.shape == (1, S, H * 128)
    seqlen = int(cu[1].item()) if (cu is not None and variant != "wan") else S
    if seqlen < n_img * 128:   # the test checks that the product leaves these rows zero as well
        assert (ref_out[0, seqlen:n_img * 128] == 0).all()

    rng = np.random.default_rng(seed)
    truth_img, txt = T._sample_blocks(n_img, tb)
    others = sorted(set(range(n_img)) - set(truth_img))
    extra = rng.choice(others, size=min(len(others), MASK_BLOCKS - len(truth_img)), replace=False) if others else []
    mask_blocks = sorted(truth_img + [int(b) for b in extra])
    img_end = min(seqlen, S)
    pairs = []
    for b in mask_blocks:
        pairs += _pairs(rng, b, TRUTH_PAIRS if b in truth_img else OTHER_PAIRS, img_end, H)
    for b in txt:
        pairs += _pairs(rng, b, TEXT_PAIRS, S, H)
    rows = np.array([p[0] for p in pairs], dtype=np.int32)
    heads = np.array([p[1] for p in pairs], dtype=np.int32)
    o = ref_out.view(S, H, 128)[torch.from_numpy(rows).long().cuda(), torch.from_numpy(heads).long().cuda()]
    mb = torch.tensor(mask_blocks, device=ref_mask.device)
    mask = ref_mask[0][:, mb].cpu().numpy()
    return {
        "fingerprint": T.fingerprint(inp),
        "mask_blocks": np.array(mask_blocks, dtype=np.int32),
        "mask": np.packbits(mask, axis=-1),
        "rows": rows, "heads": heads,
        "out": o.contiguous().view(torch.int16).cpu().numpy().view(np.uint16),
        "dtype": np.array(str(ref_out.dtype).replace("torch.", "")),
    }


def main():
    out = Path(sys.argv[1]) if len(sys.argv) > 1 else HERE / "reference_parity.npz"
    arrays = {}
    for i, case in enumerate(T.CASES):
        for key, val in case_golden(case, 1000 + i).items():
            arrays[f"{case}/{key}"] = val
        print(f"[golden] {case}: {len(arrays[f'{case}/rows'])} output pairs, "
              f"{len(arrays[f'{case}/mask_blocks'])} mask blocks", flush=True)
        torch.cuda.empty_cache()
    out.parent.mkdir(parents=True, exist_ok=True)
    np.savez_compressed(out, **arrays)
    print(f"[golden] {out} ({out.stat().st_size} bytes)")


if __name__ == "__main__":
    main()
