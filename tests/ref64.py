"""A float64 reference of the IDCT / up-sampling / colour stage and the rule decoded samples are checked against it
with.  Test infrastructure.

Input: the quantised coefficients per component in zigzag order with absolute DC (as Batch.coefficients() and the
oracle return them), each component's quantisation table (zigzag order), sampling factors, the frame size and the
up-sampling (box replication, T.81 A.2.3 / decoder.rs:347-379, or libjpeg's triangle filter as tests/fancy_ref.py).
Steps, all in float64: dequantise and de-zigzag; the exact 2-D DCT-III (transform.rs:55-87) with an 8x8 cosine matrix,
vectorised over blocks; placement; colour conversion restating decoder.rs:382-402 with the +128.  The result is the
sample BEFORE truncation.

Comparison rule (no mean-based tolerance): a decoded 8-bit sample must equal clamp(trunc(ref), 0, 255), unless ref lies
within `bound` of an integer n; then clamp(n - 1) and clamp(n) are both accepted.  `bound` is the float32 error budget
of the decoder's arithmetic for that sample:

    bound = c * 2^-24 * (S_Y + 2 * (S_Cb + S_Cr) + 256)

S_k = sum of |dequantised coefficient| over the block of component k the sample comes from (over the two or four
blocks the triangle filter reads from, the largest).  An IDCT output is at most S/4.  The decoder's factorised (AAN)
8-point passes put about ten float32 roundings on any path from a coefficient to a sample (the pre-scaled quantisation
multiplier, the butterflies of two passes), each at most 2^-24 of an intermediate no larger than about S/2; that is
some 5 * 2^-24 * S.  The colour conversion weights chroma by at most 1.772 (green's two terms by 1.06 together), hence
the factor 2, and adds three roundings of values below 256.  C_GPU = 8 covers that with margin; the largest error of
the CPU restatement of the kernels' IDCT over random blocks of every magnitude is 1.5 * 2^-24 * S.  The oracle's
direct form (transform.rs:55-87 in float32: 64-term sums of products with float32 cosines) measures 5.1 * 2^-24 * S
and gets C_ORACLE = 16.  The bound is a few float32 ulps of the magnitudes feeding the sample, so a constant off in
the fourth digit, a bias lost, or a rounding that should be a truncation leaves the band on most samples of a natural image and fails."""
import math

import numpy as np

from craft import ZIGZAG

C_GPU = 8.0
C_ORACLE = 16.0
EPS = 2.0 ** -24

_u = np.arange(8)
# transform.rs:55-87: f(x) = 1/2 sum_u alpha(u) F(u) cos((2x + 1) u pi / 16), alpha(0) = 1/sqrt(2)
COS = np.array([[(math.sqrt(0.5) if u == 0 else 1.0) * math.cos((2 * x + 1) * u * math.pi / 16) / 2 for u in _u] for x in _u])
C_RED, C_GREEN, C_BLUE = 0.299, 0.587, 0.114        # decoder.rs:392-402


class Frame:
    """What ref64 needs to know of a decoded frame.  comps: per component (coefs (n, 64) zigzag, qt (64,) zigzag,
    h, v, blocks_per_row); blocks_per_row is the MCU-padded row (mcux * h) for an interleaved scan and ceil(wc / 8)
    for a non-interleaved one."""

    def __init__(self, width, height, comps, fancy=False):
        self.width, self.height, self.fancy = width, height, fancy
        self.comps = comps
        self.hmax = max(c[2] for c in comps)
        self.vmax = max(c[3] for c in comps)


def frame_from_descriptor(d, coefs, fancy=False, scans=None):
    """A Frame from a parsed descriptor (jpeg_rust_b200.parse_descriptor) and the coefficients of its components.
    scans: instead of d, the per-component descriptors of a file with one non-interleaved scan per component
    (parse_scans); coefs then in each scan's raster block order."""
    if scans is not None:
        W, H = scans[0].frame_width, scans[0].frame_height
        hs = [s.frame_h for s in scans]
        vs = [s.frame_v for s in scans]
        hmax, vmax = max(hs), max(vs)
        comps = []
        for s, c in zip(scans, coefs):
            tq = s.comp[0].tq
            wc = -(-W * s.frame_h // hmax)
            comps.append((c, np.array(s.qt[tq][:], np.float64), s.frame_h, s.frame_v, -(-wc // 8)))
        return Frame(W, H, comps, fancy)
    W, H, n = d.width, d.height, d.ncomp
    hs = [d.comp[k].h if n > 1 else 1 for k in range(n)]
    vs = [d.comp[k].v if n > 1 else 1 for k in range(n)]
    hmax, vmax = max(hs), max(vs)
    mcux = -(-W // (8 * hmax))
    comps = []
    for k in range(n):
        c, h, v = coefs[k], hs[k], vs[k]
        if h * v > 1:       # MCU order (T.81 A.2.3: MCU by MCU, v rows of h blocks) -> raster order of the component
            c = c.reshape(-1, mcux, v, h, 64).transpose(0, 2, 1, 3, 4).reshape(-1, 64)
        comps.append((c, np.array(d.qt[d.comp[k].tq][:], np.float64), h, v, mcux * h))
    return Frame(W, H, comps, fancy)


def _component_rows(fr, k, r0, r1):
    """Samples of component k in sample rows [r0, r1) (clipped to what its blocks hold), float64, and the per-sample
    |dequantised coefficient| sums of their blocks.  Columns: all the component's sample columns."""
    coefs, qt, h, v, bpr = fr.comps[k]
    nbr = len(coefs) // bpr                      # block rows
    b0, b1 = r0 // 8, min(-(-r1 // 8), nbr)
    blk = coefs[b0 * bpr:b1 * bpr].astype(np.float64) * qt[None, :]
    nat = np.zeros_like(blk)
    nat[:, ZIGZAG] = blk                          # natural order: row = vertical frequency v, column = u
    s = np.abs(blk).sum(axis=1)
    pix = np.einsum("xu,nvu,yv->nyx", COS, nat.reshape(-1, 8, 8), COS, optimize=True)
    nb = b1 - b0
    plane = pix.reshape(nb, bpr, 8, 8).transpose(0, 2, 1, 3).reshape(nb * 8, bpr * 8)
    splane = np.repeat(np.repeat(s.reshape(nb, bpr), 8, axis=0), 8, axis=1)
    return plane[r0 - b0 * 8:r1 - b0 * 8], splane[r0 - b0 * 8:r1 - b0 * 8]


def _upsampled(fr, k, y0, y1):
    """Component k on frame rows [y0, y1), all frame columns: (value, S) float64 arrays."""
    W, H = fr.width, fr.height
    _, _, h, v, _ = fr.comps[k]
    fx, fy = fr.hmax // h, fr.vmax // v
    wc, hc = -(-W * h // fr.hmax), -(-H * v // fr.vmax)
    ys, xs = np.arange(y0, y1), np.arange(W)
    y0c = ys // fy
    if fr.fancy and fy == 2:
        yn = np.clip(y0c + np.where(ys & 1, 1, -1), 0, hc - 1)
    else:
        yn = y0c
    r0, r1 = int(min(y0c.min(), yn.min())), int(max(y0c.max(), yn.max())) + 1
    s, sa = _component_rows(fr, k, r0, r1)
    s, sa = s[:, :wc], sa[:, :wc]
    x0c = xs // fx
    xn = np.clip(x0c + np.where(xs & 1, 1, -1), 0, wc - 1) if (fr.fancy and fx == 2) else x0c
    a, c = s[np.ix_(y0c - r0, x0c)], s[np.ix_(y0c - r0, xn)]
    sab = np.maximum(np.maximum(sa[np.ix_(y0c - r0, x0c)], sa[np.ix_(y0c - r0, xn)]),
                     np.maximum(sa[np.ix_(yn - r0, x0c)], sa[np.ix_(yn - r0, xn)]))
    if fr.fancy and fy == 2:                     # libjpeg h2v2 / h1v2 fancy up-sampling: 3/4 nearer, 1/4 farther row
        a = 0.75 * a + 0.25 * s[np.ix_(yn - r0, x0c)]
        c = 0.75 * c + 0.25 * s[np.ix_(yn - r0, xn)]
    val = 0.75 * a + 0.25 * c if (fr.fancy and fx == 2) else a
    return val, sab


def bands(fr, band_rows=512, c=C_GPU):
    """Yields (y0, ref, bound): ref (rows, W, 3) float64 samples before truncation, bound (rows, W) float64, for frame
    rows [y0, y0 + rows): large frames never need their whole float64 image in memory."""
    for y0 in range(0, fr.height, band_rows):
        y1 = min(fr.height, y0 + band_rows)
        y, sy = _upsampled(fr, 0, y0, y1)
        y = y + 128.0
        if len(fr.comps) == 1:
            ref = np.repeat(y[:, :, None], 3, axis=2)
            bound = c * EPS * (sy + 256.0)
        else:
            cb, sb = _upsampled(fr, 1, y0, y1)
            cr, sr = _upsampled(fr, 2, y0, y1)
            kr, kb = 2.0 - 2.0 * C_RED, 2.0 - 2.0 * C_BLUE          # decoder.rs:392-402
            r = cr * kr + y
            b = cb * kb + y
            g = (y - C_BLUE * b - C_RED * r) / C_GREEN
            ref = np.stack([r, g, b], axis=-1)
            bound = c * EPS * (sy + 2.0 * (sb + sr) + 256.0)
        yield y0, ref, bound


def accepted(ref, bound, got):
    """Element-wise: is the 8-bit sample `got` what the rule accepts for ref (bound broadcast over channels)?
    Returns (ok, in_band)."""
    exp = np.clip(np.trunc(ref), 0, 255)
    n = np.rint(ref)
    band = np.abs(ref - n) <= bound[..., None]
    g = got.astype(np.float64)
    ok = (g == exp) | (band & ((g == np.clip(n - 1, 0, 255)) | (g == np.clip(n, 0, 255))))
    return ok, band


class Stats:
    def __init__(self):
        self.samples = self.in_band = self.bad = 0
        self.first_bad = None

    def add(self, ok, band, where=None):
        self.samples += ok.size
        self.in_band += int(band.sum())
        nbad = int(ok.size - ok.sum())
        if nbad and self.first_bad is None:
            self.first_bad = where
        self.bad += nbad

    @property
    def band_fraction(self):
        return self.in_band / max(1, self.samples)


def check_u8(fr, got_hwc, stats=None, band_rows=512, c=C_GPU):
    """Checks HxWx3 uint8 samples (RGB interleaved, or a planar output transposed) against the reference.  Returns
    Stats (bad == 0 is the pass)."""
    st = stats or Stats()
    for y0, ref, bound in bands(fr, band_rows, c):
        got = got_hwc[y0:y0 + ref.shape[0]]
        ok, band = accepted(ref, bound, got)
        if not ok.all():
            i = np.argwhere(~ok)[0]
            where = (y0 + int(i[0]), int(i[1]), int(i[2]), float(ref[tuple(i)]), int(got[tuple(i)]), float(bound[i[0], i[1]]))
        else:
            where = None
        st.add(ok, band, where)
    return st


def f32_to_u8(got_chw, scale, bias):
    """OUT_F32_PLANAR samples (3, H, W) = u8 * scale + bias per channel in float32: recovers the u8 samples and
    checks every float is that expression to within one float32 rounding of each operation."""
    scale = np.asarray(scale, np.float32).astype(np.float64)[:, None, None]
    bias = np.asarray(bias, np.float32).astype(np.float64)[:, None, None]
    g = got_chw.astype(np.float64)
    u = np.rint((g - bias) / scale)
    assert u.min() >= 0 and u.max() <= 255, (u.min(), u.max())
    want = u * scale + bias
    tol = 2.0 ** -23 * (np.abs(u * scale) + np.abs(bias) + np.abs(want))
    exact = np.abs(g - want) <= tol
    assert exact.all(), f"f32 sample is not u8 * scale + bias: {np.argwhere(~exact)[0]}"
    return u.astype(np.uint8).transpose(1, 2, 0)
