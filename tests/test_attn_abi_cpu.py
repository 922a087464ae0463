"""Argument refusals of the four attention entry points of the C ABI (include/motionclone_b200.h), called through ctypes
without a GPU: every case below is refused before the library makes any CUDA call, so the pointers are never
dereferenced."""
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from motionclone_b200 import _lib  # noqa: E402

MC_E_INVALID, MC_E_UNSUPPORTED = -1, -2
PTR = 0x10000          # 16-byte aligned, never dereferenced
MISALIGNED = 0x10008   # 8-byte aligned only


def _spatial_fwd(B=2, N=256, H=8, DH=40, ptr=PTR, null=False, stride=320):
    q = None if null else PTR
    return "spatial_attn_fwd", _lib.lib().mc_spatial_attn_fwd(
        q, PTR, PTR, ptr, None, B, N, H, DH, N * 320, stride, N * 320, 320, N * 320, 320, N * 320, 320, 0.1, None)


def _spatial_bwd(B=2, N=256, H=8, DH=40, ptr=PTR, null=False, stride=320):
    lse = None if null else PTR
    return "spatial_attn_bwd", _lib.lib().mc_spatial_attn_bwd(
        PTR, PTR, PTR, PTR, PTR, lse, ptr, PTR, PTR, PTR, B, N, H, DH, N * 320, 320, N * 320, 320, N * 320, 320,
        N * 320, 320, N * 320, 320, N * 960, stride, 0.1, None)


def _cross_fwd(B=2, Nq=1024, Nk=77, H=8, DH=40, ptr=PTR, null=False, stride=320):
    v = None if null else PTR
    return "cross_attn_fwd", _lib.lib().mc_cross_attn_fwd(
        PTR, PTR, v, ptr, B, Nq, Nk, H, DH, Nq * 320, 320, Nk * 320, stride, Nq * 320, 320, 0.1, None)


def _cross_bwd(B=2, Nq=1024, Nk=77, H=8, DH=40, ptr=PTR, null=False, stride=320):
    d_o = None if null else PTR
    return "cross_attn_bwd_dq", _lib.lib().mc_cross_attn_bwd_dq(
        PTR, PTR, PTR, d_o, ptr, B, Nq, Nk, H, DH, Nq * 320, 320, Nk * 320, 320, Nq * 320, 320, Nq * 320, stride,
        0.1, None)


ENTRIES = [_spatial_fwd, _spatial_bwd, _cross_fwd, _cross_bwd]
CASES = [
    ("null_pointer", dict(null=True), MC_E_INVALID),
    ("zero_dim", dict(H=0), MC_E_INVALID),
    ("stride_not_multiple_of_8", dict(stride=324), MC_E_INVALID),
    ("misaligned_pointer", dict(ptr=MISALIGNED), MC_E_INVALID),
    ("B_above_65535", dict(B=65536), MC_E_UNSUPPORTED),
    ("H_above_65535", dict(H=65536, DH=8), MC_E_UNSUPPORTED),
    ("head_dim_24", dict(DH=24), MC_E_UNSUPPORTED),
]


@pytest.mark.parametrize("entry", ENTRIES, ids=lambda f: f.__name__.lstrip("_"))
@pytest.mark.parametrize("case,kwargs,want", CASES, ids=[c[0] for c in CASES])
def test_attention_entry_refuses(entry, case, kwargs, want):
    name, st = entry(**kwargs)
    assert st == want, (case, st, _lib.lib().mc_last_error())
    assert _lib.lib().mc_last_error().decode().startswith(name + ":")


@pytest.mark.parametrize("entry", [_cross_fwd, _cross_bwd], ids=lambda f: f.__name__.lstrip("_"))
def test_cross_attention_refuses_more_than_80_keys(entry):
    name, st = entry(Nk=81)
    assert st == MC_E_UNSUPPORTED
    assert _lib.lib().mc_last_error().decode().startswith(name + ":")
