"""bench.py prints ONE JSON line on stdout whatever libraries write to fd 1 (NCCL prints its version
banner there on some boxes); host-side helpers of the bench (no GPU needed); --dump-outputs end to end (GPU)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_stdout_carries_only_the_json_line():
    code = (
        "import os, sys\n"
        f"sys.path.insert(0, {ROOT!r})\n"
        "import bench\n"
        "bench.own_stdout()\n"
        "os.write(1, b'NCCL version 2.28.9+cuda12.9\\n')\n"      # a C library writing to fd 1
        "print('python-level noise')\n"
        "bench.emit({'metric': 'x', 'value': 1.5})\n"
    )
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    assert json.loads(r.stdout) == {"metric": "x", "value": 1.5} and r.stdout.count("\n") == 1
    assert "NCCL version" in r.stderr and "python-level noise" in r.stderr


def test_algorithmic_work_figures():
    sys.path.insert(0, ROOT)
    import bench

    # SURVEY.md 8d: C2 GEMM flops of a fwd+bwd step (text linears x3, K/V projections x2)
    assert abs(bench.gemm_flops_per_step(8, 128, 257) / 1e9 - 990.83) < 0.01
    # decode bytes: 2 blocks x (K,V read + Q read + O written); with position rows block 0 has one query position
    D, B, Nv = 2304, 32, 257
    kv = B * 2 * Nv * D * 2
    assert bench.decode_bytes_per_step(B, 64, Nv) == 2 * (kv + 2 * B * 64 * D * 2)
    assert bench.decode_bytes_per_step(B, 64, Nv, position_rows=True) == 2 * kv + 2 * B * D * 2 * (1 + 64)
    total = sum(bench.decode_bytes_per_step(B, s, Nv) for s in range(1, 65))
    assert abs(total / 1e9 - 10.93) < 0.01


def test_decode_gemm_flops_and_workload_config():
    sys.path.insert(0, ROOT)
    import bench

    D, Dv, F, B, Nv, S = 2304, 1024, 9216, 32, 257, 64
    rows_all, rows_new = B * S * (S + 1) // 2, B * S
    per_row_rest = 2 * D * D * 4 + 4 * D * F                  # self q, k, v, o + the two FFN matrices
    per_row_cross = 2 * D * D * 2                             # w_q, w_o
    kv = 2 * 2 * (B * Nv) * Dv * D * 2                        # K and V of both blocks, once per image
    want = kv + per_row_cross * (rows_new + rows_all) + per_row_rest * 2 * rows_all
    assert bench.decode_gemm_flops(B, S, Nv) == want
    assert bench.decode_gemm_flops(B, S, Nv, position_rows=False) == want + per_row_cross * (rows_all - rows_new)
    assert abs(want / 1e12 - 18.57) < 0.01
    c1, c8 = bench.workload_config(1), bench.workload_config(8)
    assert "gradients" not in c1 and c1["parallelism"] == "single" and c1["global_batch"] == 8
    assert "bf16 arena" in c8["gradients"] and c8["parallelism"] == "dp8" and c8["global_batch"] == 64
    assert "model" not in c1 and c1["workload"].startswith("C2")


def test_dumped_outputs_are_float32_bounded_and_sampled_at_fixed_positions():
    """--dump-outputs: the loss and every gradient as float32; a large gradient is sampled at the same positions in
    every run, and the bridge's 52 gradients stay under 64 MB in all."""
    import numpy as np
    import torch

    sys.path.insert(0, ROOT)
    import bench

    assert 52 * bench.DUMP_ELEMS * 4 <= 64 << 20
    m = torch.nn.Linear(bench.DUMP_ELEMS // 256 + 1, 512)
    m(torch.randn(3, m.in_features)).square().mean().backward()
    loss = torch.tensor(1.25)
    a = bench.step_outputs(loss, m.named_parameters())
    b = bench.step_outputs(loss, m.named_parameters())
    assert sorted(a) == ["grad.bias", "grad.weight", "loss"]
    assert all(v.dtype == np.float32 for v in a.values()) and a["loss"].tolist() == [1.25]
    assert np.array_equal(a["grad.bias"], m.bias.grad.numpy())
    w = m.weight.grad.reshape(-1).numpy()
    assert a["grad.weight"].shape == (bench.DUMP_ELEMS,) and np.array_equal(a["grad.weight"], b["grad.weight"])
    assert np.isin(a["grad.weight"], w).all()


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_dump_outputs_are_identical_from_run_to_run(tmp_path):
    """bench.py --dump-outputs run twice with the same arguments writes the same arrays, in the default launch mode
    (graph replay) and under --no-graph (eager launches, which draw their dropout seeds differently)."""
    import numpy as np

    legs = ["--no-cpu-baseline", "--no-decode", "--no-train-step", "--no-inloop"]

    def run(name, *extra):
        out = tmp_path / name
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "1",
                            *legs, *extra, "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        assert json.loads(r.stdout)["steps"] == 3
        return {f: np.load(out / f) for f in sorted(os.listdir(out))}

    for extra in ((), ("--no-graph",)):
        a, b = run("a" + "".join(extra), *extra), run("b" + "".join(extra), *extra)
        assert len(a) == 53 and "loss.npy" in a and list(a) == list(b)
        assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in a.values())
        assert sum(v.nbytes for v in a.values()) <= 64 << 20
        assert [f for f in a if not np.array_equal(a[f], b[f])] == [], extra


def test_torch_library_arm_is_the_same_arithmetic():
    """bench.py's `torch_library` comparison (PyTorch's stock operators) computes the bridge: equal to the
    oracle in fp32 on the CPU at small dims, forward and gradients."""
    import torch

    sys.path.insert(0, ROOT)
    import bench
    from oracle import bridge_oracle as O

    sd = O.init_state_dict(3, vision_dim=32, language_dim=64, num_blocks=2)
    g = torch.Generator().manual_seed(1)
    for k in sd:                                             # non-trivial biases and LayerNorm affine
        if k.endswith("bias") or "ln_" in k:
            sd[k] = sd[k] + 0.1 * torch.randn(sd[k].shape, generator=g)
    vision, text = torch.randn(2, 9, 32, generator=g), torch.randn(2, 5, 64, generator=g)
    y_ref, _, dtext_ref, g_ref = O.bridge_loss_and_grads(sd, vision, text, heads_cross=2, heads_self=4)
    leaves = {k: v.clone().requires_grad_() for k, v in sd.items()}
    t = text.clone().requires_grad_()
    y = bench.torch_library_forward(leaves, vision, t, 2, 2, 4, 0.1, False)
    y.square().mean().backward()
    assert torch.allclose(y, y_ref, rtol=1e-4, atol=1e-5)
    assert torch.allclose(t.grad, dtext_ref, rtol=1e-3, atol=1e-7)
    for k in sd:
        assert torch.allclose(leaves[k].grad, g_ref[k], rtol=1e-3, atol=1e-6), k
