"""On-GPU bring-up check of the fused attention, down to decode shapes (run on the GPU machine; not a pytest file).

The row kernels, casts and column sums are covered at op level by tests/test_row_ops_gpu.py."""
from __future__ import annotations

import math
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import _harness  # noqa: E402

# ("attn", B, H, Lq, Lk, d, p)
CASES = [
    ("attn", 1, 1, 16, 32, 64, 0.0),
    ("attn", 1, 1, 64, 32, 128, 0.0),
    ("attn", 2, 3, 40, 100, 64, 0.0),
    ("attn", 2, 18, 64, 64, 128, 0.0),     # self-attention shape (C1)
    ("attn", 2, 8, 64, 257, 288, 0.0),     # cross-attention shape (C1)
    ("attn", 8, 8, 128, 257, 288, 0.0),    # C2 cross
    ("attn", 8, 18, 128, 128, 128, 0.0),   # C2 self
    ("attn", 1, 8, 5, 257, 288, 0.0),      # decode-like short prefix
    ("attn", 32, 8, 1, 257, 288, 0.0),     # C4 decode steps (K/V-streaming kernel): 1, 2, 3, 4 query row groups
    ("attn", 32, 8, 17, 257, 288, 0.0),
    ("attn", 4, 8, 33, 257, 288, 0.0),
    ("attn", 4, 8, 48, 257, 288, 0.0),
    ("attn", 32, 8, 64, 257, 288, 0.0),
    ("attn", 2, 8, 20, 5, 288, 0.0),       # one key tile: the second key split sees no key
    ("attn", 2, 18, 3, 3, 128, 0.0),       # self-attention of a 3-token prefix
    ("attn", 2, 8, 64, 1370, 288, 0.0),    # long K/V: many ring wrap-arounds
    ("attn", 2, 8, 128, 1370, 288, 0.0),   # C5 vision length
    ("attn", 2, 8, 64, 257, 288, 0.1),     # dropout
    ("attn", 2, 18, 64, 64, 128, 0.1),
]
NAMES = ["_".join(str(x) for x in c) for c in CASES]


def relerr(a, b):
    return (a.float() - b.float()).abs().max().item() / max(b.float().abs().max().item(), 1e-30)


def run_case(i: int) -> dict:
    import torch

    from vlm_bridge_b200 import ops

    c = CASES[i]
    torch.manual_seed(16 + i)   # the seeds of the recorded runs, which listed 9 row-kernel cases first
    dev = "cuda"
    res: dict = {}
    _, B, H, Lq, Lk, d, p = c
    D = H * d
    # q/k/v live inside wider fused buffers to exercise row pitches
    qb = (torch.randn(B * Lq, D + 64, device=dev)).bfloat16()
    kvb = (torch.randn(B * Lk, 2 * D, device=dev)).bfloat16()
    q, k, v = qb[:, :D], kvb[:, :D], kvb[:, D:]
    o, lse = ops.attention_fwd(q, k, v, batch=B, heads=H, len_q=Lq, len_k=Lk, head_dim=d, dropout_p=p,
                               seed=5, dropout_stream=1)
    qr = q.float().reshape(B, Lq, H, d).transpose(1, 2).requires_grad_()
    kr = k.float().reshape(B, Lk, H, d).transpose(1, 2).requires_grad_()
    vr = v.float().reshape(B, Lk, H, d).transpose(1, 2).requires_grad_()
    s = (qr @ kr.transpose(-1, -2)) / math.sqrt(d)
    pr = torch.softmax(s, -1)
    d_o = torch.randn(B * Lq, D, device=dev).bfloat16()
    dq = torch.empty(B * Lq, D, device=dev, dtype=torch.bfloat16)
    dkv = torch.empty(B * Lk, 2 * D, device=dev, dtype=torch.bfloat16)
    if p == 0:
        oref = (pr @ vr).transpose(1, 2).reshape(B * Lq, D)
        e_o = relerr(o, oref.detach())
        e_lse = (lse * math.log(2) - torch.logsumexp(s, -1)).abs().max().item()
        ops.attention_bwd(d_o, q, k, v, o, lse, dq, dkv[:, :D], dkv[:, D:], batch=B, heads=H, len_q=Lq,
                          len_k=Lk, head_dim=d)
        oref.backward(d_o.float())
        e_dq = relerr(dq, qr.grad.transpose(1, 2).reshape(B * Lq, D))
        e_dk = relerr(dkv[:, :D], kr.grad.transpose(1, 2).reshape(B * Lk, D))
        e_dv = relerr(dkv[:, D:], vr.grad.transpose(1, 2).reshape(B * Lk, D))
        res.update(e_o=e_o, e_lse=e_lse, e_dq=e_dq, e_dk=e_dk, e_dv=e_dv)
        res["ok"] = e_o < 1e-2 and e_lse < 1e-3 and e_dq < 2e-2 and e_dk < 2e-2 and e_dv < 2e-2
    else:
        # recover the mask from a run with V = identity-like probes is costly; instead check
        # (a) determinism, (b) E[o] ~ undropped o, (c) fwd/bwd mask consistency through a
        # finite-difference-free identity: with dO = o_drop-independent random, compare against a
        # torch reference that uses the mask recovered from P_drop = o when V = I (d >= Lk only).
        o2, _ = ops.attention_fwd(q, k, v, batch=B, heads=H, len_q=Lq, len_k=Lk, head_dim=d, dropout_p=p,
                                  seed=5, dropout_stream=1)
        res["deterministic"] = bool(torch.equal(o, o2))
        o0, _ = ops.attention_fwd(q, k, v, batch=B, heads=H, len_q=Lq, len_k=Lk, head_dim=d)
        res["mean_ratio"] = (o.float().abs().mean() / o0.float().abs().mean()).item()
        ok = res["deterministic"] and 0.8 < res["mean_ratio"] < 1.6
        if Lk <= d:
            # V = [I; 0] per head -> o[:, :Lk] = P_drop exactly (bf16), so the mask is observable
            eye = torch.zeros(B * Lk, D, device=dev, dtype=torch.bfloat16)
            for h in range(H):
                for j in range(Lk):
                    eye[j::Lk][:, h * d + j] = 0  # placeholder to keep shapes obvious
            ev = eye.reshape(B, Lk, H, d)
            idx = torch.arange(Lk, device=dev)
            ev[:, idx, :, idx] = 1
            ev2 = ev.reshape(B * Lk, D)
            opd, lse_d = ops.attention_fwd(q, k, ev2, batch=B, heads=H, len_q=Lq, len_k=Lk, head_dim=d,
                                           dropout_p=p, seed=5, dropout_stream=1)
            pd = opd.float().reshape(B, Lq, H, d).transpose(1, 2)[..., :Lk]   # [B,H,Lq,Lk]
            mask = (pd != 0).float()
            res["keep_frac"] = mask.mean().item()
            e_p = relerr(pd, (pr.detach() * mask / (1 - p)))
            # backward against torch autograd with that mask
            evr = ev2.float().reshape(B, Lk, H, d).transpose(1, 2).requires_grad_()
            oref = ((pr * mask / (1 - p)) @ evr).transpose(1, 2).reshape(B * Lq, D)
            ops.attention_bwd(d_o, q, k, ev2, opd, lse_d, dq, dkv[:, :D], dkv[:, D:], batch=B, heads=H,
                              len_q=Lq, len_k=Lk, head_dim=d, dropout_p=p, seed=5, dropout_stream=1)
            oref.backward(d_o.float())
            e_dq = relerr(dq, qr.grad.transpose(1, 2).reshape(B * Lq, D))
            e_dk = relerr(dkv[:, :D], kr.grad.transpose(1, 2).reshape(B * Lk, D))
            e_dv = relerr(dkv[:, D:], evr.grad.transpose(1, 2).reshape(B * Lk, D))
            res.update(e_p=e_p, e_dq=e_dq, e_dk=e_dk, e_dv=e_dv)
            ok = ok and e_p < 1e-2 and e_dq < 2e-2 and e_dk < 2e-2 and e_dv < 2e-2 and \
                abs(res["keep_frac"] - (1 - p)) < 0.02
        res["ok"] = bool(ok)
    torch.cuda.synchronize()
    return res


if __name__ == "__main__":
    sys.exit(_harness.main(os.path.abspath(__file__), NAMES, run_case, "check_ops.jsonl"))
