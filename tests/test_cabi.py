"""The C ABI without a GPU: the library builds for sm_100a, loads, exports every symbol include/*.h declares,
and rejects bad arguments before touching the device."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from gppvae_b200 import _lib, build
    build.build()
    return _lib.load(build_if_missing=False)


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "gppvae_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(gpp_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_are_exported_and_bound(lib):
    from gppvae_b200 import _lib
    declared = _declared_symbols()
    assert len(declared) >= 25
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r" T (gpp_[a-z0-9_]+)", out))
    assert set(declared) <= exported, sorted(set(declared) - exported)
    assert set(declared) == set(_lib.EXPORTED_SYMBOLS), (sorted(set(declared) ^ set(_lib.EXPORTED_SYMBOLS)))
    for name in declared:
        assert getattr(lib, name) is not None


def test_library_is_sm100a_and_torch_free(lib):
    from gppvae_b200 import _lib
    out = subprocess.run(["cuobjdump", "-lelf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    deps = subprocess.run(["ldd", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "libtorch" not in deps and "libc10" not in deps and "libpython" not in deps


def test_version_engine_and_launch_counter(lib):
    from gppvae_b200 import _lib
    assert lib.gpp_version() >= 100
    assert _lib.gemm_engine() in ("simt-fp32", "tcgen05-3xf16")
    assert _lib.launch_count() >= 0


def test_argument_validation_needs_no_device(lib):
    assert lib.gpp_gram_vtz(None, 4, None, 4, 8, 4, 4, None, 8, None, 0, None) == -1
    assert b"gram_vtz" in lib.gpp_last_error()
    assert lib.gpp_factor(None, 4, 4, None, 0, None, None, None, 0, None) == -1
    assert lib.gpp_khatri_rao_fwd(None, 1, 1, None, 1, 1, None, None, 1, None, 4, None) == -1
    assert lib.gpp_xb_nll(None, 4, None, 4, None, 4, 8, 4, 4, None, None, 4, None, None, 0, None) == -1
    # shape contract: Q and L must be multiples of 4 (the Python layer pads)
    assert lib.gpp_gram_vtz(16, 8, 16, 8, 8, 6, 4, 16, 12, 16, 1 << 20, None) == -1


def test_kr_slot_sums_planes_modes_need_no_device(lib):
    """with_x selects the part of [cnt (x) xn | slot sums] the planes hold: 0, 1 or 2, nothing else; with_x = 2 (cnt (x) xn
    alone) does not read X, so X may be NULL, and the planes it needs are P x nviews p."""
    P, p, nviews, L = 512, 128, 3, 64
    ok_ptr = 1 << 20      # 16-byte aligned, never dereferenced: every call below is rejected before a launch
    need = lib.gpp_planes_bytes(P, nviews * p)
    assert need < lib.gpp_planes_bytes(P, nviews * (p + L))
    args = lambda X, with_x, nbytes: (X, L, 1000, ok_ptr, ok_ptr, ok_ptr, P, p, nviews, L, with_x, 10, ok_ptr, nbytes,
                                      None)
    assert lib.gpp_kr_slot_sums_planes(*args(ok_ptr, 3, need)) == -1
    assert b"with_x must be 0, 1 or 2" in lib.gpp_last_error()
    assert lib.gpp_kr_slot_sums_planes(*args(None, 1, need)) == -1
    assert b"null pointer" in lib.gpp_last_error()
    assert lib.gpp_kr_slot_sums_planes(*args(None, 2, need - 1)) == -1          # X NULL passes, the size does not
    assert b"planes buffer too small" in lib.gpp_last_error()
    assert lib.gpp_kr_slot_sums_planes(*args(ok_ptr, 0, lib.gpp_planes_bytes(P, nviews * L) - 1)) == -1
    assert b"planes buffer too small" in lib.gpp_last_error()


def test_workspace_sizes_are_consistent(lib):
    for n, Q, L in [(4005, 576, 256), (100_000, 1024, 256), (1_000_000, 4096, 256), (1, 4, 4)]:
        g = lib.gpp_gram_workspace_bytes(n, Q, L)
        # whole 128 x 128 fp32 partial tiles; the tensor-core pass 1, which serves the shape where a CUDA driver is
        # present, adds 256 bytes of absmax slots to its own workspace
        tails = (0, 256) if lib.gpp_planes_supported(n, Q, L) else (0,)
        assert g > 0 and g % (128 * 128 * 4) in tails
        assert g < 2 << 30, "pass-1 split-K workspace must stay bounded"
        assert lib.gpp_factor_state_bytes(Q) >= 3 * ((Q + 63) // 64 * 64) ** 2 * 4
        assert lib.gpp_solve_workspace_bytes(Q, L) > Q * L * 4
        assert lib.gpp_xb_workspace_bytes(n, Q, L) >= n * 4
