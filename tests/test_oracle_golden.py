"""The oracle is only as good as its pin: check it against fixtures generated from the unmodified
reference module (tests/golden/make_golden.py), and against the reference itself where a copy of it
sits in oracle/_ref (oracle/make_ref.py)."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import bridge_oracle as O
from oracle import make_ref

HERE = os.path.dirname(os.path.abspath(__file__))


def _rel(a, b, floor=1e-2):
    """Frobenius error relative to max(||b||, floor). The floor matters for the cross-attention
    key bias, whose gradient is exactly zero in exact arithmetic (softmax is shift invariant), so
    both sides hold only rounding noise there."""
    return float((a - b).norm() / b.norm().clamp_min(floor))


@pytest.fixture(scope="module")
def tiny():
    z = np.load(os.path.join(HERE, "golden", "tiny_bridge.npz"))
    cfg = json.loads(bytes(z["cfg_json"]).decode())
    sd = {k[len("param/"):]: torch.from_numpy(z[k]) for k in z.files if k.startswith("param/")}
    grads = {k[len("grad/"):]: torch.from_numpy(z[k]) for k in z.files if k.startswith("grad/")}
    t = {k: torch.from_numpy(z[k]) for k in ("vision", "text", "d_out", "y", "d_text")}
    return cfg, sd, grads, t


def test_param_names_match_fixture(tiny):
    cfg, sd, _, _ = tiny
    assert list(sd.keys()) == O.param_names(cfg["num_blocks"])
    assert len(O.param_names(2)) == 52


def test_tiny_forward_matches_reference(tiny):
    cfg, sd, _, t = tiny
    y = O.bridge_forward(sd, t["vision"], t["text"], num_blocks=cfg["num_blocks"],
                         heads_cross=cfg["num_heads_cross"], heads_self=cfg["num_heads_self"])
    assert torch.allclose(y, t["y"], atol=2e-5, rtol=1e-5)


def test_tiny_backward_matches_reference(tiny):
    cfg, sd, grads, t = tiny
    _, _, d_text, g = O.bridge_loss_and_grads(sd, t["vision"], t["text"], num_blocks=cfg["num_blocks"],
                                              heads_cross=cfg["num_heads_cross"],
                                              heads_self=cfg["num_heads_self"], d_out=t["d_out"])
    assert _rel(d_text, t["d_text"]) < 1e-5
    floor = 1e-2 * max(float(v.norm()) for v in grads.values())   # w_k.bias grads are pure rounding noise
    for k in grads:
        assert _rel(g[k], grads[k], floor) < 2e-5, k


def test_tiny_cached_kv_equals_uncached(tiny):
    cfg, sd, _, t = tiny
    kw = dict(num_blocks=cfg["num_blocks"], heads_cross=cfg["num_heads_cross"], heads_self=cfg["num_heads_self"])
    kvs = O.vision_kv(sd, t["vision"], cfg["num_blocks"])
    assert torch.equal(O.bridge_forward_cached(sd, kvs, t["text"], **kw), O.bridge_forward(sd, t["vision"], t["text"], **kw))


@pytest.fixture(scope="module")
def full_fp():
    with open(os.path.join(HERE, "golden", "full_fingerprint.json")) as f:
        return json.load(f)


@pytest.fixture(scope="module")
def full_run(full_fp):
    if full_fp["torch_version"].split("+")[0] != torch.__version__.split("+")[0]:
        pytest.skip("fingerprint depends on this torch version's CPU RNG stream")
    sd = O.init_state_dict(0)
    g = torch.Generator().manual_seed(1234)
    vision = torch.randn(2, 257, 1024, generator=g)
    text = torch.randn(2, 64, 2304, generator=g)
    y, loss, d_text, grads = O.bridge_loss_and_grads(sd, vision, text)
    return sd, y, loss, d_text, grads


def test_full_init_matches_reference_rng_stream(full_fp, full_run):
    sd = full_run[0]
    assert sum(v.numel() for v in sd.values()) == full_fp["param_numel"] == 158160384
    for k, v in full_fp["param_abs_sum"].items():
        assert abs(float(sd[k].abs().sum()) - v) <= 1e-6 * v, k


def test_full_forward_fingerprint(full_fp, full_run):
    _, y, loss, _, _ = full_run
    assert abs(float(y.mean()) - full_fp["y_mean"]) < 2e-6
    assert abs(float(y.std()) - full_fp["y_std"]) < 2e-6
    assert abs(loss - full_fp["loss"]) < 1e-5
    s = full_fp["y_samples"]
    assert torch.allclose(y[0, 0, :8], torch.tensor(s["[0,0,:8]"]), atol=2e-5)
    assert torch.allclose(y[1, 63, -8:], torch.tensor(s["[1,63,-8:]"]), atol=2e-5)
    assert torch.allclose(y[1, 17, 1000:1004], torch.tensor(s["[1,17,1000:1004]"]), atol=2e-5)


def test_full_backward_fingerprint(full_fp, full_run):
    _, _, _, d_text, grads = full_run
    assert abs(float(d_text.norm()) - full_fp["d_text_norm"]) <= 1e-4 * full_fp["d_text_norm"]
    assert len(grads) == 52
    for k, v in full_fp["grad_norms"].items():
        assert abs(float(grads[k].norm()) - v) <= 2e-4 * v + 1e-9, k


@pytest.mark.skipif(make_ref.bridge_module_path() is None, reason="no copy of the reference module in oracle/_ref")
def test_against_live_reference_module():
    ref = make_ref.load_reference_bridge_module()
    cfg = dict(vision_dim=48, language_dim=96, num_blocks=3, num_heads_cross=2, num_heads_self=3)
    torch.manual_seed(5)
    m = ref.BridgeLite(dropout=0.0, **cfg).eval()
    sd = O.init_state_dict(5, vision_dim=48, language_dim=96, num_blocks=3)
    ref_sd = m.state_dict()
    assert list(ref_sd.keys()) == list(sd.keys())
    for k in sd:
        assert torch.equal(sd[k], ref_sd[k]), k      # RNG stream restated draw for draw
    g = torch.Generator().manual_seed(6)
    vision = torch.randn(3, 7, 48, generator=g)
    text = torch.randn(3, 4, 96, generator=g).requires_grad_()
    y_ref = m(vision, text)
    y_ref.square().mean().backward()
    y, _, d_text, grads = O.bridge_loss_and_grads(sd, vision, text.detach(), num_blocks=3, heads_cross=2, heads_self=3)
    assert torch.allclose(y, y_ref.detach(), atol=2e-5)
    assert _rel(d_text, text.grad) < 1e-5
    floor = 1e-2 * max(float(p.grad.norm()) for p in m.parameters())
    for n, p in m.named_parameters():
        assert _rel(grads[n], p.grad, floor) < 2e-5, n
    # bf16 emulation tracks the reference under CPU autocast to bf16 rounding noise
    with torch.no_grad(), torch.autocast("cpu", dtype=torch.bfloat16):
        y16_ref = m(vision, text.detach()).float()
    y16 = O.bridge_forward(sd, vision, text.detach(), num_blocks=3, heads_cross=2, heads_self=3, emulate_bf16=True)
    assert float((y16 - y16_ref).abs().max() / y_ref.abs().max()) < 1e-2
