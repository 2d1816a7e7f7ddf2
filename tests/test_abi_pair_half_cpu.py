"""CPU-only checks of the argument rules of the half-height pair features (one row per mated pair): the library refuses the
combinations it does not build before any CUDA call."""
import ctypes

import pytest


@pytest.fixture(scope="module")
def L():
    import __graft_entry__ as ge
    ge._load_build_module().build()          # nvcc cross-compiles sm_100a without a GPU
    import twowl_b200._lib as lib_mod
    return lib_mod


def _conv_args(L, **kw):
    fake = 1 << 20                           # aligned, never dereferenced: the checks return before any launch
    a = L.ConvArgs(Kd=64, Nd=64, out=fake, **kw)
    for s in range(a.nsrc):
        a.A[s], a.W[s] = fake, fake
    for g in range(a.ngather):
        a.T[g], a.tidx[g], a.tcoef[g] = fake, fake, fake
    return a


def test_pair_conv_a_pairs_needs_one_source(L):
    a = _conv_args(L, nsrc=2, ngather=1, M=128, a_pairs=1)
    assert L.lib.twowl_pair_conv(ctypes.byref(a), None, 0, None) == -22
    assert b"a_pairs" in L.lib.twowl_last_error()


def test_pair_conv_a_pairs_needs_an_even_row_count(L):
    a = _conv_args(L, nsrc=1, ngather=1, M=127, a_pairs=1)
    assert L.lib.twowl_pair_conv(ctypes.byref(a), None, 0, None) == -22
    assert b"a_pairs" in L.lib.twowl_last_error()


def test_seg_reduce_one_row_per_pair_refuses_a_mate_matrix(L):
    fake = 1 << 20
    a = L.SegArgs(ptr=fake, col=fake, M=10, X=fake, C=64, out=fake, out2=fake, pair_sum=2, X_mate=fake)
    assert L.lib.twowl_seg_reduce(ctypes.byref(a), None) == -22
    assert b"X_mate" in L.lib.twowl_last_error()


def test_pair_init_and_dw_gn_half_height_need_an_even_row_count(L):
    fake = 1 << 20
    assert L.lib.twowl_pair_init_fwd(fake, fake, fake, 11, 64, 1, fake, None) == -22
    assert b"pairs" in L.lib.twowl_last_error()
    rc = L.lib.twowl_pair_dw_gn(fake, fake, fake, fake, fake, fake, 0.0, 0, 0, 1, fake, fake, fake, 1, 11, 64, fake, fake, fake,
                                fake, fake, 1 << 30, None)
    assert rc == -22 and b"h_pairs" in L.lib.twowl_last_error()
