"""CPU: the sparse kernel forms a gathered row's address from a 32-bit byte stride, so cbrs_spmm_csr refuses a row
stride of 2^31 bytes or more before any launch (the check is host-only: no device pointer is dereferenced)."""
import ctypes
import os

import pytest

import __graft_entry__ as entry
from deep_cbrs_amar_renaissance_b200 import _lib as L


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(L.LIB_PATH):
        entry.build()
    return L.load()


@pytest.mark.parametrize("dtype", [L.DTYPE_F32, L.DTYPE_BF16])
def test_spmm_refuses_a_row_stride_past_32_bits(lib, dtype):
    desc = L.CsrDesc()
    desc.n_rows, desc.n_chunks, desc.chunk_edges = 1, 1, 1024
    fake = ctypes.c_void_p(0x1000)   # never dereferenced: the arguments are refused first
    ldx = (1 << 31) // 4 + 1
    rc = lib.cbrs_spmm_csr(ctypes.byref(desc), fake, ldx, fake, 128, 128, L.AGG_WEIGHTED, None, 0, dtype, None, 0, None)
    assert rc == -1
    assert b"ldx" in lib.cbrs_last_error()
