"""b200b_gemm_dual: the data gradient and the weight gradient of a Linear (autograd of bridge_module.py:98,118,
196-198,216) as one grouped persistent tcgen05 launch. A tile's arithmetic is the single-problem kernel's (same k
order), so the grouped results must be BIT-EQUAL to the two separate launches; both are also checked against fp32
torch matmuls of the same bf16 operands. With integer operands in [-4, 4] every partial sum is exact in fp32 in any
order, so there the results must also equal the fp64 reference exactly (after the bf16 rounding of bf16 outputs)."""
import pytest
import torch

pytestmark = pytest.mark.gpu

# (rows, n_out, n_in): the 2304-wide projections at C2 / C5 rows, the fused self-attention QKV, ragged sizes, and a
# shape whose weight gradient prefers 256-wide tiles (the call must fall back to two launches and still be right)
SHAPES = [(1024, 2304, 2304), (2048, 2304, 2304), (1024, 6912, 2304), (520, 2304, 2304), (1024, 264, 520),
          (48, 2304, 2304), (1024, 9216, 2304)]


# exact-integer inputs: the grouped shape, a ragged M, ragged N / K, and M below one pair tile
EXACT = [(1024, 2304, 2304), (520, 2304, 2304), (1024, 264, 520), (48, 2304, 2304)]
CASES = [s + ("gauss",) for s in SHAPES] + [s + ("exact",) for s in EXACT]


@pytest.mark.parametrize("rows,n_out,n_in,inputs", CASES,
                         ids=[f"{r}-{o}-{i}" + ("-exact" if kind == "exact" else "") for r, o, i, kind in CASES])
@pytest.mark.parametrize("wdtype", [torch.float32, torch.bfloat16])
def test_grouped_launch_is_bit_equal_to_two_launches(rows, n_out, n_in, inputs, wdtype):
    from vlm_bridge_b200 import _lib, ops

    g = torch.Generator().manual_seed(rows + n_out)
    if inputs == "exact":
        def draw(r, c, scale):
            return torch.randint(-4, 5, (r, c), generator=g).float()
    else:
        def draw(r, c, scale):
            return torch.randn(r, c, generator=g) * scale
    # dY inside a wider buffer (row pitch > n_out), as the fused QKV gradient is
    dy_buf = draw(rows, n_out + 64, 0.5).bfloat16().cuda()
    dy = dy_buf[:, :n_out]
    w = draw(n_out, n_in, 0.02).bfloat16().cuda()
    x = draw(rows, n_in, 0.5).bfloat16().cuda()
    lib = _lib.lib()
    prev = lib.b200b_gemm_set_dual(1)
    try:
        before = _lib.launch_count()
        dx1, dw1 = ops.gemm_grad_pair(dy, w, x, wgrad_dtype=wdtype)
        launches_grouped = _lib.launch_count() - before
        lib.b200b_gemm_set_dual(0)
        before = _lib.launch_count()
        dx2, dw2 = ops.gemm_grad_pair(dy, w, x, wgrad_dtype=wdtype)
        launches_split = _lib.launch_count() - before
    finally:
        lib.b200b_gemm_set_dual(prev)
    torch.cuda.synchronize()
    assert launches_split == 2 and launches_grouped in (1, 2)
    assert torch.equal(dx1, dx2) and torch.equal(dw1, dw2)
    if inputs == "exact":
        exact_dx = dy.double() @ w.double()
        exact_dw = dy.double().t() @ x.double()
        assert torch.equal(dx1, exact_dx.float().bfloat16())
        assert torch.equal(dw1, exact_dw.float().to(wdtype))
    ref_dx = dy.float() @ w.float()
    ref_dw = dy.float().t() @ x.float()
    assert float((dx1.float() - ref_dx).abs().max() / ref_dx.abs().max()) <= 1e-2
    assert float((dw1.float() - ref_dw).abs().max() / ref_dw.abs().max()) <= (1e-2 if wdtype == torch.bfloat16 else 1e-5)
    if (rows, n_out, n_in) == (1024, 2304, 2304):
        assert launches_grouped == 1          # the shape the kernel exists for really takes the grouped path
