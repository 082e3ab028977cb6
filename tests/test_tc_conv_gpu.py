"""tcgen05 3x3 convolution against a plain PyTorch fp32 reference (same bf16-rounded inputs), and, on integer inputs whose
sums are exact in any order, bit for bit against a float64 reference rounded to bf16 once."""
import ctypes

import pytest
import torch

import alphazero_chess_b200 as az

pytestmark = pytest.mark.gpu


def _run(n_boards, cin, residual, relu, iters=0, lattice=False):
    """lattice: integer inputs in [-8, 8], weights in {-1, 0, 1}, integer bias and residual: every sum is an integer below 2^14,
    exact in fp32 whatever the order of its terms, and the reference (float64) is exact before its one bf16 rounding."""
    torch.manual_seed(n_boards * 7 + cin)
    dev = "cuda:0"
    if lattice:
        x = torch.randint(-8, 9, (n_boards, 8, 8, cin), device=dev).to(torch.bfloat16)
        w = torch.randint(-1, 2, (9, 128, cin), device=dev).to(torch.bfloat16)
        bias = torch.randint(-64, 65, (128,), device=dev).float()
        res = torch.randint(-64, 65, (n_boards, 8, 8, 128), device=dev).to(torch.bfloat16) if residual else None
    else:
        x = torch.randn(n_boards, 8, 8, cin, device=dev).to(torch.bfloat16)
        w = (torch.randn(9, 128, cin, device=dev) / (3.0 * cin ** 0.5)).to(torch.bfloat16)
        bias = torch.randn(128, device=dev)
        res = torch.randn(n_boards, 8, 8, 128, device=dev).to(torch.bfloat16) if residual else None
    out = torch.full((n_boards, 8, 8, 128), float("nan"), device=dev).to(torch.bfloat16)
    ms = ctypes.c_float(0)
    L = az.lib()
    L.az_dbg_conv3x3_tc.restype = ctypes.c_int
    rc = L.az_dbg_conv3x3_tc(ctypes.c_void_p(x.data_ptr()), cin, ctypes.c_void_p(w.data_ptr()), ctypes.c_void_p(bias.data_ptr()),
                             ctypes.c_void_p(res.data_ptr() if residual else 0), ctypes.c_void_p(out.data_ptr()), n_boards,
                             int(relu), iters, ctypes.byref(ms))
    assert rc == 0, rc
    torch.cuda.synchronize()
    ft = torch.float64 if lattice else torch.float32
    wt = w.to(ft).view(3, 3, 128, cin).permute(2, 3, 0, 1).contiguous()  # [co][ci][ky][kx]
    ref = torch.nn.functional.conv2d(x.to(ft).permute(0, 3, 1, 2), wt, bias.to(ft), padding=1)
    if residual:
        ref = ref + res.to(ft).permute(0, 3, 1, 2)
    if relu:
        ref = torch.relu(ref)
    ref = ref.permute(0, 2, 3, 1)
    return out.float(), ref, ms.value


@pytest.mark.parametrize("n_boards", [1, 2, 3, 7, 299, 4096])
@pytest.mark.parametrize("cin", [128, 64, 32])
def test_conv3x3_matches_torch(n_boards, cin):
    out, ref, _ = _run(n_boards, cin, residual=True, relu=True)
    assert torch.isfinite(out).all()
    err = (out - ref).abs()
    tol = 0.02 + 0.01 * ref.abs()  # bf16 output rounding (2^-8 relative) on fp32-accumulated sums
    assert (err <= tol).all(), f"max err {err.max().item()} at {err.argmax().item()}"


_LATTICE_DBG = [(cin, dbg) for cin in (32, 64, 128) for dbg in (0, 32, 512, 64, 256, 1024)
                if dbg not in (64, 256, 1024) or (dbg == 64 and cin == 128) or (dbg == 256 and cin != 64) or (dbg == 1024 and cin == 32)]


@pytest.mark.parametrize("grid", [148, 8])
@pytest.mark.parametrize("cin,dbg", _LATTICE_DBG)
@pytest.mark.parametrize("n_boards", [1, 2, 3, 4, 5, 7, 8, 299, 4096])
def test_conv3x3_lattice_is_bit_exact(n_boards, cin, dbg, grid, monkeypatch):
    """Integer operands: the output is the reference's bf16 bits exactly, for every epilogue / box / store option
    (AZ_DBG_CONV) and for grids with several tiles per CTA (AZ_DBG_GRID=8)."""
    monkeypatch.setenv("AZ_DBG_CONV", str(dbg))
    monkeypatch.setenv("AZ_DBG_GRID", str(grid))
    out, ref, _ = _run(n_boards, cin, residual=True, relu=True, lattice=True)
    want = ref.to(torch.float32).to(torch.bfloat16)   # exact in float32 (|sum| < 2^14), then one round to nearest even
    ob, wb = out.to(torch.bfloat16).view(torch.int16), want.view(torch.int16)
    wrong = (ob != wb).nonzero()
    assert len(wrong) == 0, f"{len(wrong)} outputs differ, first at [board, row, file, channel] {wrong[0].tolist()}: " \
                            f"{out[tuple(wrong[0])].item()} vs {want[tuple(wrong[0])].item()}"


def test_conv3x3_no_residual_no_relu():
    out, ref, _ = _run(64, 128, residual=False, relu=False)
    err = (out - ref).abs()
    assert (err <= 0.02 + 0.01 * ref.abs()).all(), err.max().item()


def test_conv3x3_input_layer_speed_report():
    for cin in (64, 32):
        out, ref, ms = _run(4096, cin, residual=False, relu=True, iters=20)
        print(f"\nconv3x3 tc ({cin} padded input channels): {ms * 1e3:.1f} us @4096 boards")
        assert ms > 0


def test_conv3x3_speed_report():
    out, ref, ms = _run(4096, 128, residual=True, relu=True, iters=20)
    flops = 2.0 * 4096 * 64 * 128 * 1152
    print(f"\nconv3x3 tc: {ms * 1e3:.1f} us/layer @4096 boards -> {flops / ms / 1e9:.1f} TFLOP/s")
    assert ms > 0
