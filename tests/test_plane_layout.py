"""Executable specification of the fp16 plane layout that carries activations between the tcgen05 conv layers
(csrc/conv_split.cu) - a NumPy emulation of the index arithmetic of those kernels, checked
against torch's conv2d on the CPU:

  * plane row / swizzle addressing, hi/lo split and its round trip (what conv1 / the epilogues write and
    launch_unsplit reads back),
  * a CTA's tile = one contiguous byte range of a plane, placed at row offset g0 & 7 of a 1024-byte aligned
    buffer, read back through the absolute-address swizzle the UMMA descriptors apply (measured on B200),
  * the implicit GEMM over row-shifted tiles (9 taps) == conv2d(padding=1), positions x channels, with the
    epilogue's row <-> (segment, h, w) map, pooling and the centre-column pick of conv6.

No GPU and no library call: this pins the layout contract the CUDA kernels implement (their numerical parity is
tests/test_gpu_parity.py's job).
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

LEAD = 16            # kSplitLead (csrc/common.cuh)


class Geom(object):
    def __init__(self, H, W, C):
        self.H, self.W, self.C = H, W, C
        self.P, self.BLK, self.ROWB = W + 1, (H + 1) * (W + 1), 2 * C
        self.G, self.HALO = 256 // self.BLK, W + 2
        self.AROWS = 256 + 2 * self.HALO

    def rows(self, n_seg):
        return LEAD + n_seg * self.BLK + 256 + 32

    def row(self, seg, hh, ww):
        return LEAD + seg * self.BLK + hh * self.P + ww


def swz(off, rowb):
    """Swizzle<log2(rowb/16), 4, 3> on a byte offset (split_off / the hardware pattern)."""
    return off ^ ((off >> 3) & (rowb - 16))


def split(x):
    """split8 of csrc/tc_ptx.cuh: x >= 0 -> (hi, lo) fp16 with hi + lo == x to 2^-22."""
    x = np.minimum(x.astype(np.float32), np.float32(60000.0))
    hi = x.astype(np.float16)
    lo = (x - hi.astype(np.float32)).astype(np.float16)
    return hi, lo


def pack_planes(x, g):
    """x [seg][H][W][C] fp32 (>= 0) -> two byte planes in the HBM layout (zero rows / columns untouched)."""
    n_seg = x.shape[0]
    hi_p = np.zeros(g.rows(n_seg) * g.ROWB, np.uint8)
    lo_p = np.zeros_like(hi_p)
    hi, lo = split(x)
    for s in range(n_seg):
        for h in range(g.H):
            for w in range(g.W):
                row = g.row(s, h + 1, w + 1)
                for c8 in range(g.C // 8):
                    o = swz(row * g.ROWB + c8 * 16, g.ROWB)
                    hi_p[o:o + 16] = hi[s, h, w, c8 * 8:c8 * 8 + 8].view(np.uint8)
                    lo_p[o:o + 16] = lo[s, h, w, c8 * 8:c8 * 8 + 8].view(np.uint8)
    return hi_p, lo_p


def unpack_planes(hi_p, lo_p, g, n_seg):
    out = np.zeros((n_seg, g.H, g.W, g.C), np.float32)
    for s in range(n_seg):
        for h in range(g.H):
            for w in range(g.W):
                row = g.row(s, h + 1, w + 1)
                for c8 in range(g.C // 8):
                    o = swz(row * g.ROWB + c8 * 16, g.ROWB)
                    a = hi_p[o:o + 16].view(np.float16).astype(np.float32)
                    b = lo_p[o:o + 16].view(np.float16).astype(np.float32)
                    out[s, h, w, c8 * 8:c8 * 8 + 8] = a + b
    return out


def load_tile(plane, g, seg0):
    """The CTA's bulk copy: AROWS rows starting at plane row g0 land at row offset sh = g0 & 7 of a 1024-byte
    aligned shared-memory buffer; returns a reader (tile row r, chunk c) -> 8 halves that applies the
    descriptor's absolute-address swizzle, and sh."""
    g0 = LEAD + seg0 * g.BLK - g.HALO
    sh = g0 & 7
    smem = np.full((g.AROWS + 8) * g.ROWB, 0xFF, np.uint8)          # 0xFF..: NaN halves wherever nothing was copied
    smem[sh * g.ROWB:(sh + g.AROWS) * g.ROWB] = plane[g0 * g.ROWB:(g0 + g.AROWS) * g.ROWB]

    def read(r, c):                                                  # r: row counted from the tile's first row
        a = swz((sh + r) * g.ROWB + c * 16, g.ROWB)
        return smem[a:a + 16].view(np.float16).astype(np.float32)
    return read, sh


def tile_matrix(hi_p, lo_p, g, seg0):
    """X[r][ci] = hi + lo for the AROWS tile rows (what the MMAs see, hi and lo summed)."""
    rh, _ = load_tile(hi_p, g, seg0)
    rl, _ = load_tile(lo_p, g, seg0)
    X = np.zeros((g.AROWS, g.C), np.float64)
    for r in range(g.AROWS):
        for c8 in range(g.C // 8):
            X[r, c8 * 8:c8 * 8 + 8] = rh(r, c8).astype(np.float64) + rl(r, c8).astype(np.float64)
    return X


def implicit_gemm(X, wgt, g):
    """D[n][co] = sum_tap sum_ci X[HALO + n + off(tap)][ci] * wgt[co][ci][ky][kx], n = 0..255, tap = ky*3 + kx,
    off = (ky - 1) * P + (kx - 1)   (the row-shifted descriptor start of the kernels)."""
    D = np.zeros((256, wgt.shape[0]), np.float64)
    for t in range(9):
        ky, kx = t // 3, t % 3
        off = (ky - 1) * g.P + (kx - 1)
        D += X[g.HALO + off:g.HALO + off + 256] @ wgt[:, :, ky, kx].astype(np.float64).T
    return D


@pytest.mark.parametrize("H,W,C", [(24, 7, 16), (12, 5, 32), (12, 5, 64), (6, 3, 64), (24, 8, 16), (6, 2, 64)])
def test_planes_round_trip_and_zero_padding(H, W, C):
    g = Geom(H, W, C)
    rng = np.random.default_rng(H * 100 + W)
    x = np.abs(rng.standard_normal((3, H, W, C))).astype(np.float32) * 3
    hi_p, lo_p = pack_planes(x, g)
    back = unpack_planes(hi_p, lo_p, g, 3)
    assert np.abs(back - x).max() <= 3e-6 * max(1.0, x.max())            # 2^-22 relative
    # chunks never collide and padding positions stay zero: exactly 3*H*W*C halves are non-zero
    assert np.count_nonzero(hi_p.view(np.float16)) == np.count_nonzero(split(x)[0])
    for s in range(3):
        for hh in range(H + 1):
            for ww in range(W + 1):
                if hh == 0 or ww == 0:
                    o = g.row(s, hh, ww) * g.ROWB
                    assert not hi_p[o:o + g.ROWB].any() and not lo_p[o:o + g.ROWB].any()


@pytest.mark.parametrize("H,W,C,seg0", [(12, 5, 64, 0), (12, 5, 64, 3), (12, 5, 32, 6), (6, 3, 64, 9), (24, 7, 16, 2)])
def test_tile_is_a_contiguous_range_read_through_the_absolute_swizzle(H, W, C, seg0):
    g = Geom(H, W, C)
    n_seg = seg0 + g.G + 1
    rng = np.random.default_rng(7)
    x = np.abs(rng.standard_normal((n_seg, H, W, C))).astype(np.float32)
    hi_p, lo_p = pack_planes(x, g)
    read, sh = load_tile(hi_p, g, seg0)
    hi = split(x)[0].astype(np.float32)
    for s in range(g.G):
        for hh in range(H + 1):
            for ww in range(W + 1):
                r = g.HALO + s * g.BLK + hh * g.P + ww                  # tile row of this padded position
                for c8 in range(C // 8):
                    want = hi[seg0 + s, hh - 1, ww - 1, c8 * 8:c8 * 8 + 8] if hh and ww else np.zeros(8, np.float32)
                    np.testing.assert_array_equal(read(r, c8), want)
    # the farthest taps stay inside the copied range: rows [0, AROWS)
    assert g.HALO - g.P - 1 == 0 and g.HALO + 255 + g.P + 1 == g.AROWS - 1 and 0 <= sh < 8


CASES = [  # name, H, W, Cin, pool, pow, center, padding of the reference conv
    ("conv3A", 12, 5, 32, None, 0, False, (1, 1)),
    ("conv4A", 12, 5, 64, "adapt", 3, False, (1, 1)),
    ("conv6A", 6, 3, 64, None, 0, True, (1, 0)),
    ("conv4S", 12, 4, 64, "2x2", 2, False, (1, 1)),
]


@pytest.mark.parametrize("name,H,W,C,pool,pow_,center,pad", CASES)
def test_implicit_gemm_over_shifted_tiles_is_conv2d(name, H, W, C, pool, pow_, center, pad):
    g = Geom(H, W, C)
    rng = np.random.default_rng(11)
    n_seg = g.G + 2                                                       # second CTA is partial
    x = np.abs(rng.standard_normal((n_seg, H, W, C))).astype(np.float32)
    wgt = (rng.standard_normal((64, C, 3, 3)) * 0.1).astype(np.float32)
    bias = (rng.standard_normal(64) * 0.1).astype(np.float32)
    hi_p, lo_p = pack_planes(x, g)
    xs = torch.from_numpy(unpack_planes(hi_p, lo_p, g, n_seg)).permute(0, 3, 1, 2).double()   # what the planes hold
    ref = F.relu(F.conv2d(xs, torch.from_numpy(wgt).double(), torch.from_numpy(bias).double(), padding=pad))
    if pool == "adapt":
        ref = F.adaptive_max_pool2d(ref, (H // 2, pow_))
    elif pool == "2x2":
        ref = F.max_pool2d(ref, 2)
    ref = ref.permute(0, 2, 3, 1).numpy()                                 # [seg][h][w][c]
    w_hi = wgt.astype(np.float16)
    w_lo = (wgt - w_hi.astype(np.float32)).astype(np.float16)
    w_sum = w_hi.astype(np.float64) + w_lo.astype(np.float64)
    for cta in range((n_seg + g.G - 1) // g.G):
        seg0 = cta * g.G
        live = min(g.G, n_seg - seg0)
        X = tile_matrix(hi_p, lo_p, g, seg0)
        # conv_split.cu order: positions x channels
        D = implicit_gemm(X, w_sum, g)
        tol = 2e-5          # weights enter as w_hi + w_lo (2^-22 of |w|), accumulation in float64 here
        # conv_pipe_kernel's epilogue: thread <-> tile row r = s*BLK + hh*P + ww (interior rows only)
        for s in range(live):
            for h in range(H):
                for w in range(W):
                    if center and w != 1:
                        continue
                    r = s * g.BLK + (h + 1) * g.P + (w + 1)
                    v = np.maximum(D[r] + bias, 0.0)
                    if not pool:
                        np.testing.assert_allclose(v, ref[seg0 + s, h, 0 if center else w], rtol=0, atol=tol)
            if pool:
                # pooling epilogue of conv_pipe_kernel: max over the staged interior rows of each pooling window
                # (adaptive windows [floor(pw*W/POW), ceil((pw+1)*W/POW)) or 2x2)
                for ph in range(H // 2):
                    for pw in range(pow_):
                        x0, x1 = ((pw * W) // pow_, -(-(pw + 1) * W // pow_)) if pool == "adapt" else (2 * pw, 2 * pw + 2)
                        rows = [s * g.BLK + (hy + 1) * g.P + (x + 1) for hy in (2 * ph, 2 * ph + 1) for x in range(x0, x1)]
                        v = np.maximum(D[rows] + bias, 0.0).max(axis=0)
                        np.testing.assert_allclose(v, ref[seg0 + s, ph, pw], rtol=0, atol=tol)
