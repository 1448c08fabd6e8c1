"""GPU checks of the operand layouts of the MLP GEMMs (csrc/mlp.cu) against float64.

The weight-gradient GEMM reads both operands MN-major (dZ^T and X^T straight out of the row-major dZ and X) and
the data-gradient GEMM reads W^T MN-major out of W; the bias gradient is the column sum of dZ, reduced from
per-32-row partial sums.  A one-layer MLP with no activation isolates the two GEMMs: dx = dy W is the data
gradient, dW = dy^T x the weight gradient, db = colsum(dy).  The shapes are the layers of the default bottom
(13-512-256-128) and top (479-512-512-256-1) MLPs, at batches that do and do not fill whole 32- and 128-row
blocks, so that partial k-blocks and boxes past the end of the MN dimension are exercised."""
import ctypes

import numpy as np
import pytest
import torch

import util

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

LAYERS = [(13, 512), (512, 256), (256, 128), (479, 512), (512, 512), (512, 256)]   # (K, N) per layer


def _err(a, ref):
    ref = ref.double()
    return float((a.double() - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


class _OneLayer:
    """cdlrm_mlp object for dims [K, N] with an identity last layer (sigmoid_layer = -2)."""

    def __init__(self, K, N, cap):
        from cdlrm_b200._lib import check, lib
        self.lib, self.check = lib, check
        dims = (ctypes.c_int32 * 2)(K, N)
        need = lib.cdlrm_mlp_workspace_bytes(1, dims, cap)
        assert need > 0
        self.ws = torch.empty(need + 256, dtype=torch.uint8, device=DEV)
        base = (self.ws.data_ptr() + 255) & ~255
        self.h = ctypes.c_void_p()
        check(lib.cdlrm_mlp_create(ctypes.byref(self.h), 0, 1, dims, cap, -2, ctypes.c_void_p(base), need))

    def run(self, x, W, b, dy):
        from cdlrm_b200._lib import ptr_array
        B, K = x.shape
        N = W.shape[0]
        stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        y = torch.empty(B, N, device=DEV)
        self.check(self.lib.cdlrm_mlp_forward(self.h, ctypes.c_void_p(x.data_ptr()), x.stride(0), B,
                                              ptr_array([W.data_ptr()]), ptr_array([b.data_ptr()]),
                                              ctypes.c_void_p(y.data_ptr()), y.stride(0), stream))
        lddx = (K + 3) & ~3
        dx = torch.empty(B, lddx, device=DEV)
        dW = torch.empty(N, K, device=DEV)
        db = torch.empty(N, device=DEV)
        self.check(self.lib.cdlrm_mlp_backward(self.h, ctypes.c_void_p(dy.data_ptr()), dy.stride(0),
                                               ctypes.c_void_p(dx.data_ptr()), lddx, ptr_array([dW.data_ptr()]),
                                               ptr_array([db.data_ptr()]), stream))
        torch.cuda.synchronize()
        return y, dx[:, :K], dW, db

    def close(self):
        self.lib.cdlrm_mlp_destroy(self.h)


def _check_one_layer(K, N, B):
    g = torch.Generator(device=DEV).manual_seed(K * 1000 + N + B)
    x = torch.randn(B, K, device=DEV, generator=g)
    W = torch.randn(N, K, device=DEV, generator=g) / K ** 0.5
    b = torch.randn(N, device=DEV, generator=g)
    dy = torch.randn(B, N, device=DEV, generator=g)
    m = _OneLayer(K, N, max(B, 64))
    try:
        y, dx, dW, db = m.run(x, W, b, dy)
        _, _, _, db2 = m.run(x, W, b, dy)
    finally:
        m.close()
    x64, W64, dy64 = x.double(), W.double(), dy.double()
    refs = {"y": x64 @ W64.T + b.double(), "dx": dy64 @ W64, "dW": dy64.T @ x64, "db": dy64.sum(0)}
    for name, mine in (("y", y), ("dx", dx), ("dW", dW), ("db", db)):
        e = _err(mine, refs[name])
        assert e <= 1e-5, f"K={K} N={N} B={B} {name}: {e:.3e} off the FP64 reference"
        util.assert_close_fp32(mine.cpu().numpy(), refs[name].float().cpu().numpy(), err_msg=f"K={K} N={N} B={B} {name}")
    # the bias gradient is reduced in a fixed order: the same bits on every run
    assert torch.equal(db, db2)


@pytest.mark.parametrize("K,N", LAYERS)
def test_mn_major_gemms_at_layer_shapes(K, N):
    _check_one_layer(K, N, 8192)


@pytest.mark.parametrize("K,N,B", [
    (13, 512, 8191), (479, 512, 8191), (512, 256, 8191),
    (13, 512, 100), (479, 512, 100), (256, 128, 100),
    (13, 512, 1), (479, 512, 1),
    (479, 13, 1000),                # N = 13: one partial 32-wide column block on the MN-major side
    (13, 479, 129),                 # N = 479, one row past a 128-row tile
])
def test_mn_major_gemms_ragged(K, N, B):
    _check_one_layer(K, N, B)


def _ambiguous_rows(seq, x, thr=1e-4):
    """Rows with a ReLU pre-activation within `thr` of zero (there the mask depends on the last bits of any FP32
    forward); the caller zeroes dy on them so that gradients compare."""
    amb = torch.zeros(x.shape[0], dtype=torch.bool, device=x.device)
    h = x.double()
    mods = list(seq)
    for i, m in enumerate(mods):
        h = torch.nn.functional.linear(h, m.weight.double(), m.bias.double()) if isinstance(m, torch.nn.Linear) else m(h)
        if isinstance(m, torch.nn.Linear) and i + 1 < len(mods) and isinstance(mods[i + 1], torch.nn.ReLU):
            amb |= (h.abs() < thr).any(dim=1)
    return amb


@pytest.mark.parametrize("which,B", [("bot", 8191), ("top", 8191), ("bot", 100), ("top", 100), ("top", 1)])
def test_full_backward_weight_and_bias_gradients(which, B):
    """dW and db of every layer of a full cdlrm_mlp_backward (dgrad epilogue column sums, the split of the top
    gradient and the narrow last layer all feed db) against float64."""
    from cdlrm_b200 import model_no_ddp as M
    ln_bot, ln_top = [13, 512, 256, 128], [479, 512, 512, 256, 1]
    np.random.seed(23)
    net = M.DLRM_Net(np.asarray(ln_bot), np.asarray(ln_top), arch_interaction_op="dot", arch_interaction_itself=False,
                     sigmoid_bot=-1, sigmoid_top=len(ln_top) - 2).to(DEV)
    net.mlp_impl = "tcgen05"
    seq = net.bot_l if which == "bot" else net.top_l
    dims = ln_bot if which == "bot" else ln_top
    g = torch.Generator(device=DEV).manual_seed(B)
    x = torch.randn(B, dims[0], device=DEV, generator=g)
    dy = torch.randn(B, dims[-1], device=DEV, generator=g)
    dy[_ambiguous_rows(seq, x)] = 0.0
    seq64 = torch.nn.Sequential(*[type(m)(m.in_features, m.out_features) if isinstance(m, torch.nn.Linear) else type(m)()
                                  for m in seq]).double().to(DEV)
    seq64.load_state_dict({k: v.double() for k, v in seq.state_dict().items()})
    seq64(x.double()).backward(dy.double())
    for p in seq.parameters():
        p.grad = None
    net.apply_mlp(which, x).backward(dy)
    torch.cuda.synchronize()
    for i, (mine, p64) in enumerate(zip(seq.parameters(), seq64.parameters())):
        ref = p64.grad
        e = _err(mine.grad, ref)
        kind = "dW" if i % 2 == 0 else "db"
        assert e <= 1e-5, f"{which} B={B} layer {i // 2} {kind}: {e:.3e} off the FP64 reference"
        util.assert_close_fp32(mine.grad.cpu().numpy(), ref.float().cpu().numpy(), err_msg=f"{which} layer {i // 2} {kind}")
