"""Shared helpers for the -m gpu parity tests."""
import numpy as np
import torch


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def bits_nan_as_class(a):
    """bits() with every NaN written as 0x7FC00000.  The sign and payload of a NaN are not part of the
    result: x86 keeps an input NaN's payload and gives 0xFFC00000 for 0 * Inf, the GPU gives 0x7FFFFFFF."""
    b = bits(a).copy()
    b[np.isnan(np.asarray(a, dtype=np.float32))] = 0x7FC00000
    return b


def assert_same_bits_nan_as_class(y, ref, what=""):
    """Bit-identical results, every NaN counted as one value."""
    by, br = bits_nan_as_class(y), bits_nan_as_class(ref)
    bad = np.flatnonzero(by != br)
    assert bad.size == 0, (f"{what}: {bad.size} rows differ in their bits, first row {bad[0]}: "
                           f"{y[bad[0]]!r} (0x{by[bad[0]]:08x}) against {ref[bad[0]]!r} (0x{br[bad[0]]:08x})")


class GpuCSR:
    """Library-owned CSR (host arrays + csr_to_gpu), freed on close()."""

    def __init__(self, sp, rows, cols, rp, ci, va):
        self.sp = sp
        self.rows, self.cols = rows, cols
        self.rp, self.ci, self.va = (np.ascontiguousarray(rp, np.int32), np.ascontiguousarray(ci, np.int32),
                                     np.ascontiguousarray(va, np.float32))
        self.mat = sp.csr_from_arrays(rows, cols, self.rp, self.ci, self.va)
        rc = sp.csr_to_gpu(self.mat)
        assert rc == 0, sp.spmv_error_string(rc)

    def close(self):
        self.sp.csr_destroy(self.mat)


def run_csr(sp, A, x, kernel, dev, rows, vec_size=None):
    d_x = torch.as_tensor(np.ascontiguousarray(x, np.float32)).to(dev) if not torch.is_tensor(x) else x
    d_y = torch.full((max(rows, 1),), float("nan"), dtype=torch.float32, device=dev)
    res = sp.spmv_csr(A, d_x, d_y, sp.make_config(kernel) if kernel is not None else None,
                      len(d_x) if vec_size is None else vec_size)
    assert res.error_code == 0, (kernel, res.error_code)
    return d_y[:rows].cpu().numpy(), res


def assert_within_tolerance(y, y64, scale, what=""):
    """north_star: |y - y_ref| <= 1e-5 * sum_j |a_ij x_j| per row."""
    err = np.abs(y.astype(np.float64) - y64)
    bad = err > 1e-5 * scale + 1e-30
    assert not bad.any(), f"{what}: {bad.sum()} rows out of tolerance, worst {err[bad].max()} at row {np.argmax(bad)}"
