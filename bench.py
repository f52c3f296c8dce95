#!/usr/bin/env python
"""bench.py — carved-attention hot path at the BASELINE.json workload.

One "step" = one call of the AttenCarve operator (block pooling of q and k, block
scoring/selection, block-sparse attention incl. the dense text rows) on one DiT layer's
q,k,v at the HunyuanVideo 720x1280x125f shape: q,k,v [1, 115456, 24, 128] bf16
(900 image blocks + 2 text blocks), Jenga-Base stage-0 settings (sa-drop 0.7 -> top_k 270,
p_remain 0.3, text_amp 0, 26-neighbour adjacency of the 32x45x80 gilbert curve).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--drop 0.7]
                    [--dump-outputs DIR]

N>1 (torchrun): Ulysses — image tokens sharded over ranks outside the operator, all-to-all to
(all tokens x H/N heads) inside (jenga_b200.ulysses), strong scaling of the same layer.

value            carved-attention TFLOP/s, algorithmic FLOPs (4*128^3 per live tile from the
                 popcount of the selection mask + dense text rows) / step time, inputs
                 resident in HBM, CUDA-event timed, max over ranks.
e2e              same FLOPs / time of the same call with q,k,v in PINNED HOST memory copied
                 H2D inside the timed region and the result copied D2H.
roofline         attention kernel alone (CUDA events on its stream), vs the measured bf16
                 tensor peak in MEASURED_PEAKS.json.
cpu_baseline     the oracle port (oracle/attention_oracle.py) on the host cores, bounded sample.
--impl reference the reference's CPU-runnable path for this operator (torch SDPA with the
                 expanded block mask, hyvideo/modules/attenion.py:102-107) on a bounded sample.
--dump-outputs   writes the operator output of the last timed step as DIR/out.npy (float32; under
                 N>1 each rank's token slice as DIR/out_rank<r>.npy).  Inputs are seeded, so two
                 builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

BLOCK = 128


# ------------------------------------------------------------------------------------------------
# workload
# ------------------------------------------------------------------------------------------------
def workload(name: str, drop: float):
    if name == "hy720p":
        return dict(name="HunyuanVideo 720x1280x125f Jenga-Base layer (q,k,v [1,115456,24,128] bf16)",
                    grid=(32, 45, 80), sliced=0, heads=24, text_tokens=256, text_valid=180,
                    text_blocks=2, p_remain=0.3, drop=drop, variant="hyvideo", text_amp=0.0,
                    first_frame=0, layers=60, computed_steps=23)
    if name == "wan1.3b":
        return dict(name="Wan2.1-1.3B 832x480x81f layer (q,k,v [1,32760,12,128])",
                    grid=(21, 30, 52), sliced=1, heads=12, text_tokens=0, text_valid=0,
                    text_blocks=0, p_remain=0.9, drop=0.5, variant="wan", text_amp=0.0,
                    first_frame=(21 * 30 * 52 + 127) // 128 // 21, layers=30, computed_steps=60)
    if name == "hy_turbo_s0":  # BASELINE configs[2], stage 0 of Jenga-Turbo: 0.75x latent grid, text_amp on
        return dict(name="HunyuanVideo Jenga-Turbo stage 0 layer (grid 32x33x60, q,k,v [1,63616,24,128])",
                    grid=(32, 33, 60), sliced=0, heads=24, text_tokens=256, text_valid=180,
                    text_blocks=2, p_remain=0.3, drop=0.75, variant="hyvideo", text_amp=0.431,
                    first_frame=0, layers=60, computed_steps=12)
    if name == "hy_i2v":  # BASELINE configs[4] shape: 400 text tokens -> 4 text blocks, ragged S
        return dict(name="HunyuanVideo-I2V 720x1280x125f layer (q,k,v [1,115600,24,128])",
                    grid=(32, 45, 80), sliced=0, heads=24, text_tokens=400, text_valid=300,
                    text_blocks=4, p_remain=0.3, drop=0.75, variant="hyvideo_i2v", text_amp=0.0,
                    first_frame=0, layers=60, computed_steps=24)
    if name == "wan14b":  # BASELINE configs[3]
        return dict(name="Wan2.1-14B 1280x720x81f layer (q,k,v [1,75600,40,128])",
                    grid=(21, 45, 80), sliced=1, heads=40, text_tokens=0, text_valid=0,
                    text_blocks=0, p_remain=0.8, drop=0.7, variant="wan", text_amp=0.0,
                    first_frame=(21 * 45 * 80 + 127) // 128 // 21, layers=40, computed_steps=100)
    if name == "tiny":  # CI / smoke
        return dict(name="tiny 8x16x16 grid, 4 heads", grid=(8, 16, 16), sliced=0, heads=4,
                    text_tokens=256, text_valid=180, text_blocks=2, p_remain=0.3, drop=drop,
                    variant="hyvideo", text_amp=0.0, first_frame=0, layers=1, computed_steps=1)
    raise SystemExit(f"unknown workload {name}")


def synth_tokens(n_tokens, heads, dev, seed, gain=2.0, win=8):
    """SURVEY §8d regime P: x = 0.5 N(0,1) + gain * c[block]; c = unit vectors low-pass
    filtered along the curve order, then per-head RMS normalisation (weight 1) like the
    reference's q/k norm.  Returns [1, n_tokens, heads, 128] bf16."""
    g = torch.Generator(device=dev).manual_seed(seed)
    nb = (n_tokens + BLOCK - 1) // BLOCK
    c = torch.randn(heads, nb + win - 1, 128, generator=g, device=dev)
    c = torch.nn.functional.avg_pool1d(c.transpose(1, 2), win, 1).transpose(1, 2)[:, :nb]
    c = c / c.norm(dim=-1, keepdim=True)
    out = torch.empty(1, n_tokens, heads, 128, dtype=torch.bfloat16, device=dev)
    chunk = 64
    for b0 in range(0, nb, chunk):
        b1 = min(nb, b0 + chunk)
        r0, r1 = b0 * BLOCK, min(n_tokens, b1 * BLOCK)
        x = 0.5 * torch.randn(heads, (b1 - b0) * BLOCK, 128, generator=g, device=dev)
        x = x + gain * c[:, b0:b1].repeat_interleave(BLOCK, dim=1)
        x = x[:, : r1 - r0]
        x = x * torch.rsqrt(x.pow(2).mean(-1, keepdim=True) + 1e-6)
        out[0, r0:r1] = x.transpose(0, 1).to(torch.bfloat16)
    return out


def build_inputs(wl, dev, heads=None, seed=1234):
    from jenga_b200 import gilbert
    t, h, w = wl["grid"]
    heads = heads or wl["heads"]
    n_img = t * h * w
    S = n_img + wl["text_tokens"]
    q = synth_tokens(S, heads, dev, seed)
    k = synth_tokens(S, heads, dev, seed + 1)
    v = torch.randn(1, S, heads, 128, generator=torch.Generator(device=dev).manual_seed(seed + 2),
                    device=dev).to(torch.bfloat16)
    nbr = gilbert.block_neighbor_mapping(t, h, w, sliced=bool(wl["sliced"]))
    nb_img = (n_img + BLOCK - 1) // BLOCK
    if wl["variant"] == "wan":
        top_k = math.ceil(int(nb_img * (1 - wl["drop"])))       # wan/modules/model_mul.py:162-164
        cu = None
        q, k = q.float(), k.float()  # rope_apply returns .float() (wan/modules/model_mul.py:71)
    else:
        top_k = int((1 - wl["drop"]) * (n_img // BLOCK))          # models_mul…:242
        cu = torch.tensor([0, n_img + wl["text_valid"], S], dtype=torch.int32, device=dev)
    return dict(q=q, k=k, v=v, nbr=nbr, top_k=top_k, cu=cu, S=S, n_img=n_img, nb_img=nb_img,
                heads=heads)


def run_operator(wl, inp, q=None, k=None, v=None, return_bits=False):
    from jenga_b200.attention import block_sparse_attention_variant
    q = inp["q"] if q is None else q
    k = inp["k"] if k is None else k
    v = inp["v"] if v is None else v
    return block_sparse_attention_variant(
        wl["variant"], q, k, v, inp["top_k"], cu_seqlens_q=inp["cu"], cu_seqlens_kv=inp["cu"],
        text_blocks=wl["text_blocks"], text_amp=wl["text_amp"], block_neighbor_list=inp["nbr"],
        p_remain_rates=wl["p_remain"], first_frame_blocks=wl["first_frame"],
        return_mask_bits=return_bits)


def algorithmic_flops(wl, inp, bits):
    """4*128*128*128 per live (q-block, k-block) tile + dense text rows (BASELINE.md FLOP rule)."""
    words = bits.to(torch.int64) & 0xFFFFFFFF
    pop = 0
    x = words
    # popcount via byte table-free bit tricks
    x = x - ((x >> 1) & 0x5555555555555555)
    x = (x & 0x3333333333333333) + ((x >> 2) & 0x3333333333333333)
    x = (x + (x >> 4)) & 0x0F0F0F0F0F0F0F0F
    pop = int(((x * 0x0101010101010101) >> 56 & 0xFF).sum().item())
    tile = 4 * BLOCK * BLOCK * 128
    text_rows = wl["text_blocks"] * BLOCK
    nb_all = (inp["S"] + BLOCK - 1) // BLOCK
    dense = 4 * inp["heads"] * text_rows * nb_all * BLOCK * 128
    return pop * tile + dense, pop


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.samples, self._stop, self._t = index, [], threading.Event(), None

    def _loop(self):
        while not self._stop.is_set():
            try:
                r = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                    "-i", str(self.index)], capture_output=True, text=True, timeout=5)
                if r.returncode == 0 and r.stdout.strip():
                    self.samples.append([s.strip() for s in r.stdout.strip().split(",")])
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._t = threading.Thread(target=self._loop, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit())
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            for n, val in zip(names, s[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": float(self.samples[0][1]) if self.samples[0][1].replace(".", "").isdigit() else None,
                "power_w_max": max((float(s[2]) for s in self.samples if s[2].replace(".", "").isdigit()), default=None),
                "samples": len(self.samples), "reasons": sorted(reasons)}


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return dict(bf16_burst=d.get("bf16_tflops", 1590.0), bf16_sustained=d.get("bf16_tflops_sustained", 1400.0),
                    hbm=d.get("hbm_gbs", 6650.0), source="measured (MEASURED_PEAKS.json)")
    return dict(bf16_burst=1590.0, bf16_sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


# ------------------------------------------------------------------------------------------------
# CPU legs — bounded samples of the SAME workload on the host cores.
#   kind "sdpa-port": the reference's CPU-runnable path for this operator, torch SDPA with the
#                     expanded block mask (hyvideo/modules/attenion.py:102-107,
#                     wan/modules/attention.py:167-176), on the workload's REAL selection mask
#                     (oracle builder on the same synthetic tokens) for a sample of query blocks.
#   kind "port":      the oracle's tile loop (oracle/attention_oracle.carved_attention_rows).
# Both use every host core (torch.set_num_threads(os.cpu_count())) and report it.
# ------------------------------------------------------------------------------------------------
_CPU_CASE = {}


def _cpu_case(wl, nq):
    """One head of the workload on the CPU: tokens, the oracle-built mask rows of `nq` evenly spaced
    query blocks, and their live-tile count."""
    key = (wl["name"], wl["drop"], nq)
    if key in _CPU_CASE:
        return _CPU_CASE[key]
    from oracle import attention_oracle as orc
    from jenga_b200 import gilbert
    t, h, w = wl["grid"]
    n_img = t * h * w
    S = n_img + wl["text_tokens"]
    nb = (S + BLOCK - 1) // BLOCK
    tb = wl["text_blocks"]
    n_img_b = nb - tb
    cpu = torch.device("cpu")
    q = synth_tokens(nb * BLOCK, 1, cpu, 1234)[:, :, 0].unsqueeze(1)   # [1,1,Sp,128] bf16
    k = synth_tokens(nb * BLOCK, 1, cpu, 1235)[:, :, 0].unsqueeze(1)
    v = torch.randn(1, 1, nb * BLOCK, 128, generator=torch.Generator().manual_seed(1236)).bfloat16()
    if S < nb * BLOCK:
        for x in (q, k, v):
            x[:, :, S:] = 0
    nbr = gilbert.block_neighbor_mapping(t, h, w, sliced=bool(wl["sliced"]))
    if wl["variant"] == "wan":
        top_k = math.ceil(int(n_img_b * (1 - wl["drop"])))
    else:
        top_k = int((1 - wl["drop"]) * (n_img // BLOCK))
    mask = orc.build_block_onehot(q[:, :, :n_img_b * BLOCK], k, top_k, n_img_b, nb, wl["p_remain"], tb, nbr,
                                  wl["first_frame"])                       # [1,1,n_img_b,nb]
    rows = sorted({int(round(i * (n_img_b - 1) / max(nq - 1, 1))) for i in range(nq)})
    qs = torch.cat([q[:, :, r * BLOCK:(r + 1) * BLOCK] for r in rows], dim=2)
    ms = mask[:, :, rows]
    seqlen = n_img + wl["text_valid"] if wl["variant"] != "wan" else S
    _CPU_CASE[key] = dict(q=qs, k=k, v=v, mask=ms, rows=rows, live=int(ms.sum()), S=S, nb=nb, n_img_b=n_img_b,
                          seqlen=seqlen)
    return _CPU_CASE[key]


def cpu_sample(wl, kind: str, nq: int, min_seconds: float):
    """Returns (TFLOP/s algorithmic, sample description, seconds per rep, threads)."""
    from oracle import attention_oracle as orc
    ncores = os.cpu_count() or 1
    torch.set_num_threads(ncores)
    c = _cpu_case(wl, nq)
    flops = 4 * BLOCK * BLOCK * 128 * c["live"]
    reps, t_total = 0, 0.0
    while reps == 0 or t_total < min_seconds:
        t0 = time.perf_counter()
        if kind == "port":
            orc.carved_attention_rows(c["q"], c["k"], c["v"], c["mask"], c["seqlen"], 128 ** -0.5, wl["text_amp"],
                                      c["n_img_b"])
        else:
            big = c["mask"].repeat_interleave(BLOCK, 2).repeat_interleave(BLOCK, 3)
            big[..., c["seqlen"]:] = False
            torch.nn.functional.scaled_dot_product_attention(c["q"], c["k"], c["v"], attn_mask=big)
        t_total += time.perf_counter() - t0
        reps += 1
    tf = flops * reps / t_total / 1e12
    sample = (f"1 head x {len(c['rows'])} query blocks (evenly spaced) x their {c['live']} live key tiles of the "
              f"workload's own mask (nb={c['nb']}, S={c['S']}), {reps} reps, {t_total:.1f}s, "
              f"{torch.get_num_threads()} threads")
    return tf, sample, t_total / reps, torch.get_num_threads()


# ------------------------------------------------------------------------------------------------
# GPU reference leg: the UNMODIFIED reference operator (Triton JIT + FlashAttention-2) on the same
# tensors on the same B200 (SURVEY §8d "Reference timed beside it (1)").  Checker/baseline only.
# ------------------------------------------------------------------------------------------------
def gpu_reference_leg(wl, inp, iters=3):
    sys.path.insert(0, str(ROOT / "tests"))
    try:
        from oracle import ref_loader
        import refutil
        if not ref_loader.available():
            return {"unavailable": "oracle/_ref/ not staged (run __graft_entry__.build() where /root/reference is mounted)"}
        op = ref_loader.operator(wl["variant"])
    except Exception as e:  # noqa: BLE001
        return {"unavailable": f"{type(e).__name__}: {e}"}
    q, k, v, cu, nbr = inp["q"], inp["k"], inp["v"], inp["cu"], inp["nbr"]
    S = inp["S"]
    nb = (S + BLOCK - 1) // BLOCK
    tb = wl["text_blocks"]
    n_img = nb - tb
    kw = dict(top_k=inp["top_k"], text_blocks=tb, nbr=nbr, p_remain=wl["p_remain"], first_frame=wl["first_frame"])
    nbr_dev = nbr.to(q.device)  # the reference moves it lazily on first use (:282-283); keep that out of the timing
    kw["nbr"] = nbr_dev

    def total():
        return refutil.reference_call(op, wl["variant"], q, k, v, cu=cu, text_amp=wl["text_amp"], **kw)

    def timed(fn, n):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            r = fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n, r

    try:
        for _ in range(3):  # first call includes the Triton JIT
            total()
        total_ms, _ = timed(total, iters)
        mask_ms, mask = timed(lambda: refutil.reference_mask(op, wl["variant"], q, k, **kw), iters)
        # the two kernels alone, on the layouts block_sparse_attention_combined hands them
        qh, kh, vh = (refutil.pad_rows(x, nb * BLOCK).transpose(1, 2) for x in (q, k, v))
        if wl["variant"] == "wan":
            qh, kh, vh = (x.to(torch.bfloat16) for x in (qh, kh, vh))
        seq = (cu[1:2].to(torch.int32) if (cu is not None and wl["variant"] != "wan")
               else torch.tensor([S], dtype=torch.int32, device=q.device))
        triton_ms, _ = timed(lambda: op._triton_block_sparse_attention_onehot(
            qh[:, :, :n_img * BLOCK], kh, vh, seq, mask, 128 ** -0.5, BLOCK, BLOCK, is_text_block=False,
            text_amp=wl["text_amp"], text_block_start=n_img), iters)
        fa2_ms = None
        if tb > 0:
            fa2_ms, _ = timed(lambda: op.flash_attn_func(
                qh[:, :, n_img * BLOCK:].permute(0, 2, 1, 3), kh.permute(0, 2, 1, 3), vh.permute(0, 2, 1, 3),
                causal=False, softmax_scale=128 ** -0.5), iters)
        pop = int(mask.sum().item())
        flops = pop * 4 * BLOCK * BLOCK * 128 + 4 * inp["heads"] * tb * BLOCK * nb * BLOCK * 128
        isa = None
        try:
            kern = op._triton_block_sparse_attn_fwd_kernel_onehot
            for cache in getattr(kern, "device_caches", {}).values():
                for ck in cache[0].values():
                    ptx = ck.asm.get("ptx", "")
                    isa = {"tcgen05.mma": ptx.count("tcgen05.mma"), "mma.sync": ptx.count("mma.sync"),
                           "wgmma": ptx.count("wgmma"), "cp.async.bulk": ptx.count("cp.async.bulk")}
        except Exception:  # noqa: BLE001
            pass
        return {"impl": "unmodified reference block_sparse_attention (Triton %s JIT + flash_attn %s)" % (
                    __import__("triton").__version__, __import__("flash_attn").__version__),
                "total_ms": total_ms, "mask_ms": mask_ms, "triton_ms": triton_ms, "fa2_ms": fa2_ms,
                "live_tiles": pop, "tflops": flops / (total_ms * 1e-3) / 1e12,
                "triton_kernel_tflops": pop * 4 * BLOCK * BLOCK * 128 / (triton_ms * 1e-3) / 1e12,
                "triton_ptx_mma": isa, "iters": iters, "autocast": "bf16"}
    except Exception as e:  # noqa: BLE001
        return {"unavailable": f"{type(e).__name__}: {str(e)[:300]}"}


# ------------------------------------------------------------------------------------------------
# DiT block-stack leg: the UNMODIFIED reference block classes (MMDoubleStreamBlock /
# MMSingleStreamBlock, random-init at the HunyuanVideo width) run (A) with the reference's own
# operator (Triton + FA2) and (B) through jenga_b200.install (operator + fused prologue + gather
# hooks), same weights, same inputs, same GPU.  This is the measured DiT-loop number: one computed
# denoising step = 20 double + 40 single blocks (jenga_hyvideo.py:132-178); a video = 23 of them.
# ------------------------------------------------------------------------------------------------
def dit_forward_leg(wl, inp, n_double, n_single, hidden=3072, heads=24, fp8_too=False):
    try:
        from oracle import ref_loader
        if not ref_loader.available():
            return {"unavailable": "oracle/_ref/ not staged"}
        ref_hy, _ = ref_loader.load_blocks(product=False)
        our_hy, _ = ref_loader.load_blocks(product=True)
    except Exception as e:  # noqa: BLE001
        return {"unavailable": f"{type(e).__name__}: {e}"}
    from jenga_b200 import blocks as jb
    from jenga_b200 import gilbert
    dev = inp["q"].device
    t, h, w = wl["grid"]
    L, T = inp["n_img"], wl["text_tokens"]
    g = torch.Generator(device=dev).manual_seed(2024)

    def init(m):
        with torch.no_grad():
            for n_, p_ in m.named_parameters():
                if p_.dim() >= 2:
                    p_.copy_(torch.randn(p_.shape, generator=g, device=dev, dtype=torch.float32).mul_(0.02))
                elif "norm" in n_:
                    p_.fill_(1.0)
                else:
                    p_.zero_()

    def stack(mod):
        d = [mod.MMDoubleStreamBlock(hidden, heads, mlp_width_ratio=4.0, dtype=torch.bfloat16, device=dev)
             for _ in range(n_double)]
        s_ = [mod.MMSingleStreamBlock(hidden, heads, mlp_width_ratio=4.0, dtype=torch.bfloat16, device=dev)
              for _ in range(n_single)]
        return d, s_

    try:
        rd, rs = stack(ref_hy)
        for b_ in rd + rs:
            init(b_)
        with torch.device("meta"):
            od = [our_hy.MMDoubleStreamBlock(hidden, heads, mlp_width_ratio=4.0, dtype=torch.bfloat16) for _ in range(n_double)]
            os_ = [our_hy.MMSingleStreamBlock(hidden, heads, mlp_width_ratio=4.0, dtype=torch.bfloat16) for _ in range(n_single)]
        for a_, b_ in zip(od + os_, rd + rs):
            a_.load_state_dict(b_.state_dict(), assign=True)     # shared weights, no second copy
        l2h, h2l = gilbert.mapping_tensors(t, h, w)
        l2h, h2l = l2h.to(dev), h2l.to(dev)
        curve_sel = [[l2h, h2l, inp["nbr"]]]
        img0 = torch.randn(1, L, hidden, generator=g, device=dev).bfloat16()
        txt0 = torch.randn(1, T, hidden, generator=g, device=dev).bfloat16()
        vec = torch.randn(1, hidden, generator=g, device=dev).bfloat16()
        ang = torch.rand(L, 64, generator=g, device=dev) * 6.2831853
        cos = torch.cos(ang).repeat_interleave(2, dim=1).contiguous()
        sin = torch.sin(ang).repeat_interleave(2, dim=1).contiguous()
        cu = inp["cu"]
        drop = wl["drop"]

        def forward(dbl, sgl, hooks):
            """the block loop of ra_forward (jenga_hyvideo.py:116-118,132-178,226)"""
            if hooks:
                jb.install_gather_hook()
            else:
                jb.remove_gather_hook()
            img = img0[:, h2l]
            fc, fs = cos[h2l], sin[h2l]
            txt = txt0
            for blk in dbl:
                img, txt = blk(img, txt, vec, cu, cu, L + T, L + T, (fc, fs), drop, wl["text_amp"], curve_sel, wl["p_remain"])
            x = torch.cat((img, txt), 1)
            for blk in sgl:
                x = blk(x, vec, T, cu, cu, L + T, L + T, (fc, fs), drop, wl["text_amp"], curve_sel, wl["p_remain"])
            return x[:, :L][:, l2h]

        def timed(fn, n):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                r = fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) * 1e-3 / n, r

        nblk = n_double + n_single
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            forward(rd[:1], rs[:1], False)                                    # Triton JIT + cuBLAS warm-up
            ref_s, ref_out = timed(lambda: forward(rd, rs, False), 1)
            forward(od, os_, True)
            our_s, our_out = timed(lambda: forward(od, os_, True), 2)
        fp8_s = None
        if fp8_too:   # opt-in FP8 P.V variant, reported separately, never the headline
            from jenga_b200 import attention as _A
            _A.PV_FP8 = True
            try:
                with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
                    forward(od, os_, True)
                    fp8_s, fp8_out = timed(lambda: forward(od, os_, True), 2)
            finally:
                _A.PV_FP8 = False
        jb.remove_gather_hook()
        rms = ref_out.float().pow(2).mean().sqrt().item()
        diff = (our_out.float() - ref_out.float()).abs()
        scale = (20 + 40) / nblk
        return {"blocks_measured": {"double": n_double, "single": n_single}, "hidden": hidden, "heads": heads,
                "reference_seconds": ref_s, "ours_seconds": our_s, "speedup": ref_s / our_s,
                "seconds_per_computed_step": {"reference": ref_s * scale, "ours": our_s * scale,
                                              "note": "measured blocks x (60 / measured), blocks are homogeneous"},
                "dit_loop_sec_per_video": {"reference": ref_s * scale * wl["computed_steps"],
                                           "ours": our_s * scale * wl["computed_steps"],
                                           "computed_steps": wl["computed_steps"]},
                "output_vs_reference": {"max_over_rms": diff.max().item() / rms, "mean_over_rms": diff.mean().item() / rms},
                "fused_calls": {k_: v_ for k_, v_ in jb.STATS.items()},
                **({"optin_fp8_pv": {"ours_seconds": fp8_s, "speedup": ref_s / fp8_s,
                                     "output_vs_reference_mean_over_rms": (fp8_out.float() - ref_out.float()).abs().mean().item() / rms,
                                     "note": "JENGA_PV_FP8=1: e4m3 P and V in the second product; lower precision, not the headline"}}
                   if fp8_s else {}),
                "what": "unmodified reference block classes, random-init bf16 weights; A = reference operator "
                        "(Triton+FA2), B = the same classes through jenga_b200.install hooks"}
    except Exception as e:  # noqa: BLE001
        import traceback
        return {"unavailable": f"{type(e).__name__}: {str(e)[:300]}", "trace": traceback.format_exc()[-600:]}


DUMP_LIMIT_BYTES = 48_000_000   # what all dumped files may add up to, with room for .npy headers


def dump_output(out: torch.Tensor, path: Path, limit: int = DUMP_LIMIT_BYTES) -> None:
    """Writes `out` ([1, rows, ...], one row per token) as float32 .npy.  An output over `limit`
    bytes is reduced to a fixed sample of whole rows (seeded, sorted, the same for every run of
    the same shape)."""
    import numpy as np
    x = out.detach().reshape(out.shape[1], -1)
    rows, cols = x.shape
    keep = max(1, min(rows, limit // (4 * cols)))
    if keep < rows:
        idx = torch.randperm(rows, generator=torch.Generator().manual_seed(0))[:keep].sort().values
        x = x[idx.to(x.device)]
    path.parent.mkdir(parents=True, exist_ok=True)
    np.save(path, x.float().cpu().numpy())


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="hy720p")
    ap.add_argument("--drop", type=float, default=0.7)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dit-loop", type=int, default=0, metavar="STEPS",
                    help="also run the step-skip schedule harness for this many computed steps "
                         "(23 = the whole 50-step video: 1380 hot-path calls) and report measured "
                         "hot-path seconds per video")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dit-blocks", default="4,8",
                    help="DiT block-stack leg: 'D,S' double,single blocks to build and time for both the "
                         "reference and this library (default 4,8 = 1/5 of a forward; 'full' = 20,40; 'none')")
    ap.add_argument("--pv-fp8", action="store_true",
                    help="ALSO time the opt-in FP8 P.V variant (reported under 'fp8_pv_variant'; never the headline)")
    ap.add_argument("--no-gpu-reference", action="store_true",
                    help="skip timing the unmodified reference operator (Triton + FA2) on this GPU")
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path,
                    help="write the operator output of the last timed step to DIR/out.npy (float32; a "
                         "fixed sample of its rows when it exceeds 48 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    wl = workload(args.workload, args.drop)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    metric = "carved_attn_tflops"
    if args.impl == "reference":
        if rank != 0:
            return
        nq = int(os.environ.get("JENGA_REF_NQ", "32"))
        for _ in range(max(1, min(args.warmup, 2))):
            cpu_sample(wl, "sdpa-port", nq, 0.0)
        vals = []
        for _ in range(max(1, args.steps)):
            tf_i, sample, sec, ncores = cpu_sample(wl, "sdpa-port", nq, 3.0)   # one step >= 3 s of CPU work
            vals.append((tf_i, sec))
        tf = sum(v[0] for v in vals) / len(vals)
        ms = 1e3 * sum(v[1] for v in vals) / len(vals)
        line = {"impl": "reference", "metric": metric, "value": tf, "unit": "TFLOP/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": wl["name"], "sa_drop": wl["drop"], "p_remain": wl["p_remain"],
                           "text_blocks": wl["text_blocks"], "parallelism": "host cpu",
                           "sample": f"bounded: 1 head x {nq} query blocks of the workload's own mask, >= 3 s per step"},
                "cpu_baseline": {"value": tf, "unit": "TFLOP/s", "cores": ncores, "kind": "sdpa-port",
                                 "sample": "torch SDPA + expanded block mask (the reference's CPU-runnable path, "
                                           "hyvideo/modules/attenion.py:102-107): " + sample},
                "e2e": {"value": tf, "unit": "TFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (jenga_b200 has no CPU path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    if world > 1:
        from jenga_b200 import ulysses
        state = ulysses.bench_setup(wl, build_inputs, dev, rank, world)
        step = lambda: ulysses.bench_step(wl, state)  # noqa: E731
        inp = state["inp"]
    else:
        inp = build_inputs(wl, dev)
        step = lambda: run_operator(wl, inp)  # noqa: E731

    # FLOPs from the selection mask of this exact input (reported with the number)
    if world > 1:
        flops, pop = ulysses.bench_flops(wl, state, algorithmic_flops)
    else:
        _, bits = run_operator(wl, inp, return_bits=True)
        flops, pop = algorithmic_flops(wl, inp, bits)
    torch.cuda.synchronize()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clk:
        ev0.record()
        for _ in range(args.steps):
            last = step()
        ev1.record()
        barrier()
    ms = ev0.elapsed_time(ev1) / args.steps
    if args.dump_outputs:
        # rows: under N>1 this rank's share of the budget, so that the ranks' files stay within it
        dump_output(last, args.dump_outputs / ("out.npy" if world == 1 else f"out_rank{rank}.npy"),
                    DUMP_LIMIT_BYTES // world)
    del last
    if dist is not None:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    clocks = clk.summary()

    # ---- roofline: the attention kernel alone, CUDA events on its stream (N=1 path shape)
    roof = None
    pk = peaks()
    if world == 1:
        from jenga_b200 import attention as A
        _, bits = run_operator(wl, inp, return_bits=True)
        mask_source = "this library's selection kernels"
        r_flops, r_pop = flops, pop
        if not args.no_gpu_reference:
            # SURVEY §8d: the attention kernel is timed on the mask the REFERENCE builder produces for
            # these inputs (checker-side code, oracle/ref_loader.py); popcounts of both are reported
            try:
                sys.path.insert(0, str(ROOT / "tests"))
                from oracle import ref_loader
                import refutil
                if ref_loader.available():
                    rm = refutil.reference_mask(ref_loader.operator(wl["variant"]), wl["variant"], inp["q"], inp["k"],
                                                top_k=inp["top_k"], text_blocks=wl["text_blocks"], nbr=inp["nbr"].to(dev),
                                                p_remain=wl["p_remain"], first_frame=wl["first_frame"])
                    bits = A.mask_onehot_to_bits(rm)
                    r_flops, r_pop = algorithmic_flops(wl, inp, bits)
                    mask_source = f"reference builder (popcount {r_pop}; this library's selection: {pop})"
                    del rm
            except Exception as e:  # noqa: BLE001
                mask_source += f" (reference builder unavailable: {type(e).__name__})"
        S, nb_img = inp["S"], inp["nb_img"]
        aq, ak = (x if x.dtype == torch.bfloat16 else x.bfloat16() for x in (inp["q"], inp["k"]))
        out = torch.empty_like(aq)
        seq = inp["cu"][1:2].contiguous() if inp["cu"] is not None else None
        def attn_only():
            A._launch(aq, ak, inp["v"], bits, nb_img, wl["text_blocks"], 128 ** -0.5, wl["text_amp"],
                      nb_img, S, S, ((S + 127) // 128) * 128, out, seq, torch.bfloat16)
        for _ in range(3):
            attn_only()
        torch.cuda.synchronize()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n_it = max(5, args.steps)
        a0.record()
        for _ in range(n_it):
            attn_only()
        a1.record()
        torch.cuda.synchronize()
        ams = a0.elapsed_time(a1) / n_it
        ach = r_flops / (ams * 1e-3) / 1e12
        traffic = None
        tp = ROOT / "profiles" / "attn_traffic.json"
        if tp.exists() and args.workload == "hy720p":
            try:
                traffic = json.loads(tp.read_text()).get("dram_bytes_per_launch")
            except Exception:
                traffic = None
        roof = {"bound": "tensor", "kernel": "carved_attn_fwd_kernel", "achieved": ach, "peak": pk["bf16_burst"],
                "unit": "TFLOP/s", "frac": ach / pk["bf16_burst"], "traffic": traffic, "ms_per_launch": ams,
                "frac_of_sustained_peak": ach / pk["bf16_sustained"], "sustained_peak": pk["bf16_sustained"],
                "peak_source": pk["source"] + ", bf16 burst (kernel timed alone)",
                "algorithmic_flops_per_launch": r_flops, "live_tiles": r_pop, "mask_source": mask_source}

    # ---- e2e: host buffers, H2D + D2H inside the timed region
    e2e = None
    if not args.no_e2e and world == 1:
        # q,k,v start in pinned host memory and the result ends in pinned host memory, every step.
        # Public API: jenga_b200.host_pipeline.HostPipelinedAttention — the operator is per-head
        # independent, so head groups are staged H2D / computed / drained D2H on three streams.
        from jenga_b200.host_pipeline import HostPipelinedAttention
        # (wan: q,k are staged as bf16 here; the device-resident `value` leg keeps the fp32 inputs)
        hq, hk, hv = (x.to(torch.bfloat16).cpu().pin_memory() for x in (inp["q"], inp["k"], inp["v"]))
        hout = torch.empty_like(hq).pin_memory()
        groups = int(os.environ.get("JENGA_E2E_GROUPS", "0")) or (
            12 if inp["heads"] % 12 == 0 else (4 if inp["heads"] % 4 == 0 else 1))  # measured: 12 groups best at H=24
        pipe = HostPipelinedAttention(1, inp["S"], inp["heads"], 128, torch.bfloat16, dev, groups=groups,
                                      variant=wl["variant"])
        kw = dict(cu_seqlens_q=inp["cu"], cu_seqlens_kv=inp["cu"], text_blocks=wl["text_blocks"],
                  text_amp=wl["text_amp"], block_neighbor_list=inp["nbr"], p_remain_rates=wl["p_remain"],
                  first_frame_blocks=wl["first_frame"])
        def e2e_step():
            pipe(hq, hk, hv, hout, inp["top_k"], wait=False, **kw)   # consecutive steps overlap; finish() closes the region
        for _ in range(2):
            e2e_step()
        pipe.finish()
        torch.cuda.synchronize()
        ref_out = run_operator(wl, inp, q=inp["q"].to(torch.bfloat16), k=inp["k"].to(torch.bfloat16))
        ref_out = ref_out.view(1, inp["S"], inp["heads"], 128)
        torch.cuda.synchronize()
        e2e_ok = bool(torch.equal(hout, ref_out.cpu()))
        n_it = max(3, min(args.steps, 10))
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        b0.record()
        for _ in range(n_it):
            e2e_step()
        pipe.finish()         # every step's result is back in pinned host memory before the clock stops
        b1.record()
        torch.cuda.synchronize()
        ems = b0.elapsed_time(b1) / n_it
        e2e = {"value": flops / (ems * 1e-3) / 1e12, "unit": "TFLOP/s", "ms_per_step": ems,
               "h2d_bytes_per_step": sum(x.numel() * x.element_size() for x in (hq, hk, hv)),
               "d2h_bytes_per_step": hout.numel() * hout.element_size(),
               "api": f"host_pipeline.HostPipelinedAttention(groups={groups}), consecutive steps overlapped",
               "matches_device_resident_result": e2e_ok}
        del hq, hk, hv, hout, pipe, ref_out

    if not args.no_e2e and world > 1:
        # every rank stages ITS token slice (all heads) + the replicated text rows from pinned host
        # memory, runs the sequence-parallel operator and returns its slice of the result to the host
        hq, hk, hv = (state[n].cpu().pin_memory() for n in ("q", "k", "v"))
        n_rows = state["q"].shape[1]
        hout = torch.empty((1, n_rows, inp["heads"], 128), dtype=torch.bfloat16).pin_memory()
        e2e_api = None
        if state["mode"].startswith("fused"):
            # public API: ulysses.HostPipelinedUlysses — H2D / peer-store exchange / attention / D2H of
            # consecutive head sub-groups on four streams, copy-in running ahead into the next step
            pipe = ulysses.HostPipelinedUlysses(state["n_loc"], n_rows - state["n_loc"], inp["heads"], 128,
                                                torch.bfloat16, dev, fused=state["sp"])
            kw_ = dict(top_k=state["top_k"], text_amp=wl["text_amp"], block_neighbor_list=inp["nbr"],
                       p_remain_rates=wl["p_remain"], cu_seqlens_q=state["cu"], cu_seqlens_kv=state["cu"])
            def e2e_step():
                pipe(hq, hk, hv, hout, wait=False, **kw_)   # consecutive steps overlap; finish() closes the region
            e2e_api = f"ulysses.HostPipelinedUlysses ({pipe.G} head sub-groups per rank, 4 streams, steps overlapped; max over ranks)"
        else:
            dq, dk, dv = (torch.empty_like(state[n]) for n in ("q", "k", "v"))
            def e2e_step():
                dq.copy_(hq, non_blocking=True)
                dk.copy_(hk, non_blocking=True)
                dv.copy_(hv, non_blocking=True)
                st2 = dict(state, q=dq, k=dk, v=dv)
                hout.view(1, n_rows, -1).copy_(ulysses.bench_step(wl, st2), non_blocking=True)
            e2e_api = "ulysses.my_parallel_attention (NCCL) on per-rank pinned host slices (max over ranks)"
        e2e_finish = (lambda: pipe.finish()) if state["mode"].startswith("fused") else (lambda: None)
        for _ in range(2):
            e2e_step()
        e2e_finish()
        barrier()
        e2e_ok = None
        if state["mode"].startswith("fused"):
            want = ulysses.bench_step(wl, state).view(1, n_rows, inp["heads"], 128)
            torch.cuda.synchronize()
            e2e_ok = bool(torch.equal(hout, want.cpu()))
            tt = torch.tensor([1 if e2e_ok else 0], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MIN)
            e2e_ok = bool(tt.item())
        n_it = max(3, min(args.steps, 10))
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        b0.record()
        for _ in range(n_it):
            e2e_step()
        e2e_finish()          # every step's result is back in pinned host memory before the clock stops
        b1.record()
        barrier()
        ems = b0.elapsed_time(b1) / n_it
        t = torch.tensor([ems], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ems = t.item()
        e2e = {"value": flops / (ems * 1e-3) / 1e12, "unit": "TFLOP/s", "ms_per_step": ems,
               "h2d_bytes_per_step": world * sum(x.numel() * x.element_size() for x in (hq, hk, hv)),
               "d2h_bytes_per_step": world * hout.numel() * hout.element_size(),
               "api": e2e_api, "matches_device_resident_result": e2e_ok}

    dit = None
    if args.dit_loop > 0 and world == 1 and wl["variant"] == "hyvideo":
        from jenga_b200 import dit_loop
        L, T, H = inp["n_img"], wl["text_tokens"], inp["heads"]
        g = torch.Generator(device=dev).manual_seed(77)
        img_qkv = torch.empty(1, L, 3 * H * 128, dtype=torch.bfloat16, device=dev)
        # q,k parts: the model-like synthetic tokens (pre-norm scale 1.5), v part: N(0,1)
        img_qkv.view(1, L, 3, H, 128)[:, :, 0] = inp["q"][:, :L] * 1.5
        img_qkv.view(1, L, 3, H, 128)[:, :, 1] = inp["k"][:, :L] * 1.5
        img_qkv.view(1, L, 3, H, 128)[:, :, 2] = inp["v"][:, :L]
        txt_qkv = torch.randn(1, T, 3 * H * 128, generator=g, device=dev).to(torch.bfloat16)
        ws = [torch.ones(128, dtype=torch.bfloat16, device=dev) for _ in range(4)]
        ang = torch.rand(L, 64, generator=g, device=dev) * 6.2831853
        cos = torch.cos(ang).repeat_interleave(2, dim=1).contiguous()
        sin = torch.sin(ang).repeat_interleave(2, dim=1).contiguous()
        dit_loop.run_hot_path_loop(img_qkv, txt_qkv, H, ws, (cos, sin), inp["nbr"], inp["cu"],
                                   p_remain=wl["p_remain"], max_computed_steps=1)  # warm-up: 60 calls
        sec, calls = dit_loop.run_hot_path_loop(img_qkv, txt_qkv, H, ws, (cos, sin), inp["nbr"], inp["cu"],
                                                p_remain=wl["p_remain"], sa_drop_rates=(args.drop, min(args.drop + 0.1, 0.95)),
                                                max_computed_steps=args.dit_loop)
        n_sched = sum(1 for s_ in dit_loop.schedule() if s_[1])
        dit = {"computed_steps_run": args.dit_loop, "computed_steps_per_video": n_sched, "calls": calls,
               "seconds": sec, "hot_path_sec_per_video": sec * n_sched / args.dit_loop,
               "ms_per_call": 1e3 * sec / calls,
               "includes": "attention_prologue (RMSNorm+RoPE+cat+pool) + select_blocks + carved attention; "
                           "DiT dense layers out of scope"}
        del img_qkv, txt_qkv

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        tf, sample, _, ncores = cpu_sample(wl, "sdpa-port", int(os.environ.get("JENGA_REF_NQ", "32")), 3.0)   # same sample as --impl reference
        cpu = {"value": tf, "unit": "TFLOP/s", "cores": ncores, "kind": "sdpa-port",
               "sample": "torch SDPA + expanded block mask (same function as --impl reference): " + sample}

    ditf = None
    if rank == 0 and world == 1 and args.dit_blocks != "none" and wl["variant"] == "hyvideo" and not args.no_gpu_reference:
        nd, ns = (20, 40) if args.dit_blocks == "full" else (int(v_) for v_ in args.dit_blocks.split(","))
        torch.cuda.empty_cache()
        ditf = dit_forward_leg(wl, inp, nd, ns, fp8_too=args.pv_fp8)
        torch.cuda.empty_cache()

    fp8v = None
    if rank == 0 and world == 1 and args.pv_fp8 and wl["variant"] != "wan":
        from jenga_b200.attention import block_sparse_attention_variant as _bsa
        kw8 = dict(cu_seqlens_q=inp["cu"], cu_seqlens_kv=inp["cu"], text_blocks=wl["text_blocks"], text_amp=wl["text_amp"],
                   block_neighbor_list=inp["nbr"], p_remain_rates=wl["p_remain"], first_frame_blocks=wl["first_frame"])
        def step8():
            return _bsa(wl["variant"], inp["q"], inp["k"], inp["v"], inp["top_k"], pv_fp8=True, **kw8)
        for _ in range(3):
            step8()
        torch.cuda.synchronize()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(args.steps):
            o8 = step8()
        f1.record()
        torch.cuda.synchronize()
        ms8 = f0.elapsed_time(f1) / args.steps
        o16 = run_operator(wl, inp)
        d = (o8.float() - o16.float()).abs()
        rms = o16.float().pow(2).mean().sqrt().item()
        fp8v = {"ms_per_step": ms8, "tflops_equivalent": flops / (ms8 * 1e-3) / 1e12, "speedup_vs_bf16_path": ms / ms8,
                "vs_bf16_path": {"max_over_rms": d.max().item() / rms, "mean_over_rms": d.mean().item() / rms},
                "note": "opt-in, lower precision in P.V only (e4m3 P and V, per-head V scale); includes the two V quantisation passes"}

    gref = None
    if rank == 0 and world == 1 and not args.no_gpu_reference:
        gref = gpu_reference_leg(wl, inp)
        if "total_ms" in gref:
            gref["speedup_of_this_operator"] = gref["total_ms"] / ms

    if rank == 0:
        value = flops / (ms * 1e-3) / 1e12
        # our kernels per step: block_pool x2, pooled_scores_mma, select_rows, carved_attn (+ ulysses_scatter
        # and the same per head sub-group under Ulysses)
        launches = 5 if world == 1 else 1 + 5
        line = {
            "metric": metric, "value": value, "unit": "TFLOP/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": wl["name"], "sa_drop": wl["drop"], "top_k": inp["top_k"],
                       "p_remain": wl["p_remain"], "text_blocks": wl["text_blocks"],
                       "live_tiles": pop, "algorithmic_tflop_per_step": flops / 1e12,
                       "l2": f"inputs ({3 * inp['S'] * inp['heads'] * 256 / 1e9:.1f} GB) larger than L2, no flush",
                       "parallelism": "1 gpu" if world == 1 else f"ulysses{world} ({state['mode']})",
                       "hot_path_sec_per_video": ms * 1e-3 * wl["layers"] * wl["computed_steps"]},
            "clocks": clocks, "gpu_launches": launches * args.steps,
        }
        if e2e:
            line["e2e"] = e2e
        if roof:
            line["roofline"] = roof
        if cpu:
            line["cpu_baseline"] = cpu
        if dit:
            line["dit_loop"] = dit
        if fp8v:
            line["fp8_pv_variant"] = fp8v
        if ditf:
            line["dit_forward"] = ditf
        if gref:
            line["gpu_reference"] = gref
            line["vs_gpu_reference"] = gref.get("speedup_of_this_operator")
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
