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


def test_featmap_and_taylor_validation_needs_no_device(lib):
    """The feature-map and Taylor entries reject shapes their kernels cannot take before any launch: p + q past the
    48 KB of staged table rows, p q or a design width not a multiple of 4, ldv % 4 != 0, k outside 1..16, ldg < p q."""
    from gppvae_b200._lib import host_i32, host_i64, host_ptrs
    ok = 1 << 20          # 16-byte aligned, never dereferenced: every call below is rejected before a launch
    kr = lambda p, q, ldv: lib.gpp_khatri_rao_fwd(ok, 10, p, ok, 10, q, ok, ok, 100, ok, ldv, None)
    assert kr(1533, 4, 1533 * 4) == -1 and b"too large" in lib.gpp_last_error()          # p + q = 1537
    assert kr(3, 3, 12) == -1 and b"multiple of 4" in lib.gpp_last_error()
    assert kr(4, 3, 14) == -1 and b"ldv" in lib.gpp_last_error()
    assert kr(4, 3, 8) == -1                                                                # ldv < p q
    kp = lambda p, q, ldv: lib.gpp_khatri_rao_fwd_planes(ok, 10, p, ok, 10, q, ok, ok, 600, ok, ldv, ok, 1 << 30, ok,
                                                         1 << 30, None)
    assert kp(3, 3, 12) == -1 and b"bad shape" in lib.gpp_last_error()
    assert kp(4, 3, 14) == -1 and b"ldv" in lib.gpp_last_error()
    assert lib.gpp_khatri_rao_bwd(ok, 11, ok, 10, 4, ok, 10, 3, ok, ok, 100, ok, ok, None) == -1   # ldg < p q
    assert b"bad shape" in lib.gpp_last_error()
    assert lib.gpp_normalize_rows_fwd(ok, 10, 0, ok, None) == -1
    assert lib.gpp_normalize_rows_bwd(ok, ok, 10, 0, ok, None) == -1
    te = lambda L, Q, ldv: lib.gpp_taylor_expansion_fwd(ok, 8, ok, 8, ok, ldv, ok, 12, 100, L, Q, ok, ok, ok, None)
    assert te(6, 4, 12) == -1 and te(8, 9, 12) == -1 and b"bad shape" in lib.gpp_last_error()
    assert te(8, 8, 10) == -1 and b"ld" in lib.gpp_last_error()
    tb = lambda L, Q: lib.gpp_taylor_expansion_bwd(ok, ok, 8, ok, 12, 100, L, Q, ok, ok, ok, 8, ok, 12, ok, None)
    assert tb(6, 4) == -1 and tb(8, 9) == -1
    for k in (0, 17):
        ptrs, lds, Qs = host_ptrs([ok] * 17), host_i64([8] * 17), host_i32([8] * 17)
        assert lib.gpp_taylor_expansion_fwd_multi(ok, 8, ok, 8, k, ptrs, lds, ptrs, lds, Qs, 100, 8, ok, ok, ok,
                                                  None) == -1
        assert b"designs" in lib.gpp_last_error()
        assert lib.gpp_taylor_expansion_bwd_multi(ok, ok, 8, k, ptrs, lds, Qs, 100, 8, ok, ok, ok, 8, ptrs, lds, ok,
                                                  None) == -1
        assert b"designs" in lib.gpp_last_error()
    ptrs, lds, Qs = host_ptrs([ok] * 2), host_i64([8, 8]), host_i32([8, 6])
    assert lib.gpp_taylor_expansion_fwd_multi(ok, 8, ok, 8, 2, ptrs, lds, ptrs, lds, Qs, 100, 8, ok, ok, ok, None) == -1
    assert b"design 1 has 6 columns" in lib.gpp_last_error()
    assert lib.gpp_taylor_expansion_bwd_multi(ok, ok, 8, 2, ptrs, lds, Qs, 100, 8, ok, ok, ok, 8, ptrs, lds, ok,
                                              None) == -1
    assert b"design 1 has 6 columns" in lib.gpp_last_error()
    assert lib.gpp_split_planes_stacked(2, ptrs, lds, Qs, 600, 0, ok, 1 << 30, ok, 1 << 30, None) == -1
    assert b"design 1 has 6 columns" in lib.gpp_last_error()


def test_host_entry_validation_needs_no_device(lib):
    """The host-buffer entry and gpp_factor_solve reject bad arguments before they touch the context or the device: a
    null context, tickets other than 0 and 1, a null required pointer, p q or L not a multiple of 4, p q >= 2^30,
    Q % 4 != 0 and ldgc < Q + L or ldgc % 4 != 0."""
    import ctypes
    ok = 1 << 20          # 16-byte aligned, never dereferenced: every call below is rejected before any use
    tk = ctypes.c_int32(-7)
    ptrs = dict(ctx=ok, x0=ok, v0=ok, d=ok, w=ok, X=ok, lvs=ok, nll=ok)

    def submit(P=100, p=16, q=8, n=1000, L=64, ticket=True, **null):
        a = {k: (None if k in null else v) for k, v in ptrs.items()}
        return lib.gpp_gp_term_host_submit(a["ctx"], a["x0"], P, p, a["v0"], q, q, a["d"], a["w"], a["X"], n, L, a["lvs"],
                                           a["nll"], ok, ok, ctypes.byref(tk) if ticket else None)

    for k in ptrs:
        assert submit(**{k: True}) == -1 and b"null pointer" in lib.gpp_last_error(), k
    assert submit(ticket=False) == -1 and b"null pointer" in lib.gpp_last_error()
    assert tk.value == -7, "a rejected submission set the ticket"
    assert submit(p=3, q=3) == -1 and b"multiples of 4" in lib.gpp_last_error()
    assert submit(L=6) == -1 and b"multiples of 4" in lib.gpp_last_error()
    assert submit(p=1 << 15, q=1 << 15) == -1 and b"multiples of 4" in lib.gpp_last_error()     # p q = 2^30
    for bad in dict(P=0), dict(p=0), dict(q=0), dict(n=0), dict(L=0):
        assert submit(**bad) == -1 and b"bad shape" in lib.gpp_last_error(), bad
    assert lib.gpp_gp_term_host(None, ok, 100, 16, ok, 8, 8, ok, ok, ok, 1000, 64, ok, ok, ok, ok) == -1
    for t in (-1, 2):
        assert lib.gpp_gp_term_host_wait(ok, t) == -1 and b"bad ticket" in lib.gpp_last_error()
    assert lib.gpp_gp_term_host_wait(None, 0) == -1
    assert lib.gpp_host_ctx_create(None) == -1
    assert lib.gpp_host_ctx_destroy(None) == 0
    fs = lambda Q, L, ldgc: lib.gpp_factor_solve(ok, ldgc, Q, L, ok, 100, 0, ok, L, None, ok, ok, 1 << 30, None)
    assert fs(6, 4, 12) == -1 and b"bad shape" in lib.gpp_last_error()
    assert fs(8, 6, 16) == -1 and b"bad shape" in lib.gpp_last_error()
    assert fs(8, 4, 8) == -1 and b"bad GC" in lib.gpp_last_error()           # ldgc < Q + L
    assert fs(8, 4, 14) == -1 and b"bad GC" in lib.gpp_last_error()          # ldgc % 4 != 0
    assert lib.gpp_vbs(None, 100, 8, 4, ok, None) == -1 and lib.gpp_vbs(ok, 0, 8, 4, ok, None) == -1
