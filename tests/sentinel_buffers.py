"""Device buffers with sentinels around the matrix a kernel reads or writes, for the C-ABI kernel tests.

Inputs sit in NaN: a stray read poisons the result.  Outputs a kernel adds into sit in a finite value that is compared
bit for bit afterwards: a reduce-add or atomicAdd onto NaN leaves NaN, so a NaN sentinel cannot show a stray add.
Every address a kernel is handed stays inside the allocation.
"""
import torch

NAN = float("nan")
OUT_SENTINEL = -777.25   # exact in every floating type; any add of a non-zero value changes its bits

_BITS = {torch.float64: torch.int64, torch.float32: torch.int32, torch.bfloat16: torch.int16,
         torch.float16: torch.int16}


def same_bits(a, b):
    """a and b hold the same bit patterns (NaN equals NaN of the same payload, -0 differs from +0)."""
    return a.shape == b.shape and torch.equal(a.contiguous().view(_BITS[a.dtype]), b.contiguous().view(_BITS[b.dtype]))


class Padded:
    """A rows x cols matrix with row pitch ld inside an allocation filled with `sentinel`: `lead` elements before it,
    the pad columns cols..ld-1 of every row and `guard` whole rows after it.  `m` is the matrix view; without `fill`
    it holds the sentinel too."""

    def __init__(self, rows, cols, ld, dtype, fill=None, lead=0, guard=2, sentinel=NAN):
        n = lead + (rows + guard) * ld
        self.buf = torch.full((n,), sentinel, dtype=dtype, device="cuda")
        self.m = self.buf[lead:lead + rows * ld].view(rows, ld)[:, :cols]
        if fill is not None:
            self.m.copy_(fill)
        self.ld = ld
        self.sentinel = sentinel
        inside = torch.zeros(n, dtype=torch.bool, device="cuda")
        inside[lead:lead + rows * ld].view(rows, ld)[:, :cols] = True
        self._outside = ~inside

    @property
    def ptr(self):
        return self.m.data_ptr()

    def sentinels_intact(self):
        out = self.buf[self._outside]
        return same_bits(out, torch.full_like(out, self.sentinel))


class Segmented:
    """nseg segments of seg_rows rows (row pitch ldx, segment s starting seg_stride elements after segment s - 1) inside
    a NaN-filled allocation, the layout of a row slice h[:, a:b] of a (B, N, D) activation.  `rows` is the
    (nseg * seg_rows) x d matrix they describe."""

    def __init__(self, x, seg_rows, ldx, seg_stride, lead=0):
        rows, d = x.shape
        nseg = rows // seg_rows
        assert nseg * seg_rows == rows and seg_stride >= seg_rows * ldx and ldx >= d
        self.buf = torch.full((lead + nseg * seg_stride + ldx,), NAN, dtype=x.dtype, device="cuda")
        view = self.buf.as_strided((nseg, seg_rows, d), (seg_stride, ldx, 1), lead)
        view.copy_(x.view(nseg, seg_rows, d))
        self.rows = view.reshape(rows, d)
        self.ptr = view.data_ptr()

    def sentinels_intact(self):
        """Everything outside the segments is still NaN."""
        return bool(torch.isnan(self.buf).sum() == self.buf.numel() - self.rows.numel())
