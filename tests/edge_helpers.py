"""Helpers of the elementwise fp64 tests (test_gpu_kernel_edges.py, test_gpu_structured_kernel_edges.py): error
constants per engine, inputs with NaN in their leading-dimension gap, sentinel output buffers and the grading against
an fp64 bound.  A plain module (no tests): importing it needs no device."""
import math

import torch

U = 2.0 ** -24
FLOOR = 2.0 ** -31
NAN_BITS = 0x7FC0DEAD          # a quiet NaN with a payload no kernel produces
DEV = torch.device("cuda:0")


def stream():
    return torch.cuda.current_stream().cuda_stream


def workspace(nbytes):
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=DEV)


def call(status, what):
    from gppvae_b200 import _lib
    _lib.check(status, what)


def c_tc(k, epi=0):
    """Relative error constant of a k-long tensor-core product (3-term fp16 split; test_gpu_kernel_edges.py)."""
    return (12 + 48 + math.ceil(k / 64) + 1 + epi) * U


def c_simt(k, epi=0):
    """Relative error constant of a k-long fp32 SIMT product."""
    return (k + 1 + epi) * U


def gamma(k):
    """gamma_k = k u / (1 - k u): the relative error of a k-step fp32 recursive sum (inf when k u >= 1)."""
    return k * U / (1.0 - k * U) if k * U < 1.0 else float("inf")


def spread_cols(n, c, seed, positive=True):
    """n x c float32 with column scales log-uniform in [1e-3, 1e3]; the first eighth of the columns all-positive."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    X = torch.randn(n, c, generator=g, device=DEV)
    if positive:
        X[:, : max(1, c // 8)].abs_()
    return X * 10.0 ** (torch.rand(c, generator=g, device=DEV) * 6.0 - 3.0)


def strided(M, pad):
    """M itself (pad = 0) or a view of a wider tensor whose `pad` extra columns hold NaN; returns (view, ld)."""
    if pad == 0:
        return M.contiguous(), M.shape[1]
    n, c = M.shape
    w = torch.full((n, c + pad), float("nan"), device=DEV)
    w[:, :c] = M
    return w[:, :c], c + pad


def sentinel(rows, cols):
    """(rows + 1) x (cols + 8) float32 filled with the NaN pattern; returns (buffer, ld)."""
    return torch.full((rows + 1, cols + 8), NAN_BITS, dtype=torch.int32, device=DEV).view(torch.float32), cols + 8


def check_sentinel(buf, rows, cols, what, allow_nan=False):
    """The rows x cols block of a sentinel buffer, after checking that nothing outside it was written (and, unless
    allow_nan, that the block holds no NaN)."""
    bits = buf.view(torch.int32)
    assert bool((bits[:rows, cols:] == NAN_BITS).all()), f"{what}: wrote into the gap columns past {cols}"
    assert bool((bits[rows] == NAN_BITS).all()), f"{what}: wrote past row {rows}"
    if not allow_nan:
        assert not bool(torch.isnan(buf[:rows, :cols]).any()), f"{what}: NaN inside the {rows} x {cols} output"
    return buf[:rows, :cols]


def nan_vector(n):
    return torch.full((n + 1,), NAN_BITS, dtype=torch.int32, device=DEV).view(torch.float32)


def ratio_of(err, lim):
    r = torch.where(lim > 0, err / torch.where(lim > 0, lim, torch.ones_like(lim)),
                    torch.where(err > 0, torch.full_like(err, float("inf")), torch.zeros_like(err)))
    return float(r.max()) if r.numel() else 0.0


def grade(what, C, R, mag, floor, c):
    """Assert |C - R| <= c mag + floor elementwise; print and return the worst ratio."""
    assert bool(torch.isfinite(C).all()), f"{what}: non-finite output"
    r = ratio_of((C.double() - R).abs(), c * mag + floor)
    print(f"[{what}] worst bound ratio {r:.3f}")
    assert r <= 1.0, f"{what}: elementwise error {r:.3g} x the fp64 bound"
    return r


def atb_terms(A, B, maxB_cols=None):
    """R = A^T B, |A|^T |B| and the scale floor, in fp64 (maxB_cols: per-column maximum of B's operand scale)."""
    A64, B64 = A.double(), B.double()
    aA, aB = A64.abs(), B64.abs()
    mB = aB.max() if maxB_cols is None else maxB_cols
    floor = FLOOR * (aA.max() * aB.sum(0)[None, :] + (mB[None, :] if maxB_cols is not None else mB) * aA.sum(0)[:, None])
    return A64.t() @ B64, aA.t() @ aB, floor


def am_terms(A, M):
    A64, M64 = A.double(), M.double()
    aA, aM = A64.abs(), M64.abs()
    floor = FLOOR * (aA.max() * aM.sum(0)[None, :] + aM.max() * aA.sum(1)[:, None])
    return A64 @ M64, aA @ aM, floor
