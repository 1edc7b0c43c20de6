"""Every decoded sample of the CUDA path against the float64 reference (ref64.py) built from the GPU's own
coefficients, under ref64's rule (a decoded sample is clamp(trunc(ref)) unless ref lies within a few float32 ulps of
the magnitudes feeding it of an integer): all fused IDCT/colour variants across tile-boundary shapes, all three
output formats, the compose path, images too large for the oracle, random batches, and the crafted extremes of
craft.py (coefficients and statuses against the oracle)."""
import random
import time

import numpy as np
import pytest

import craft
import oracle_ffi as O
import ref64
from jpeg_rust_b200 import (EXT_DRI, EXT_NONE, LAYOUT_SPEC, LAYOUT_SPEC_FANCY, Batch, _ffi, decode_scans, parse_descriptor,
                            parse_scans, synth)

pytestmark = pytest.mark.gpu

WIDTHS = [1, 7, 8, 9, 15, 16, 17, 127, 128, 129, 255, 256, 257, 383, 385, 639, 641]
HEIGHTS = [1, 8, 9, 15, 16, 17, 31, 33]
SUBS = ["gray", "444", "422", "440", "420"]
SCALE = np.array([1 / 57.0, 1 / 64.3, 1 / 59.9], np.float32)      # non-identity per-channel normalisation
BIAS = np.array([-2.1, -1.7, 0.25], np.float32)


def frame_of(data, coefs, ext=EXT_DRI, fancy=False):
    st, d, _ = parse_descriptor(data, ext, LAYOUT_SPEC)
    assert st == 0
    return ref64.frame_from_descriptor(d, coefs, fancy=fancy)


def check_images(files, coefs, outs, what, stats, fancy=False, fmt=_ffi.OUT_RGB_INTERLEAVED):
    for i, f in enumerate(files):
        o = outs[i]
        if fmt == _ffi.OUT_RGB_PLANAR:
            o = o.transpose(1, 2, 0)
        elif fmt == _ffi.OUT_F32_PLANAR:
            o = ref64.f32_to_u8(o, SCALE, BIAS)
        st = ref64.check_u8(frame_of(f, coefs[i], fancy=fancy), o, stats=ref64.Stats())
        assert st.bad == 0, f"{what} image {i}: {st.bad} samples outside the rule, first (y, x, ch, ref, got, bound) {st.first_bad}"
        stats.samples += st.samples
        stats.in_band += st.in_band


def decode(files, layout=LAYOUT_SPEC):
    b = Batch(files, layout=layout, ext=EXT_DRI)
    b.upload().decode()
    outs = b.download()
    st, _ = b.results()
    assert all(s == 0 for s in st), [(i, s) for i, s in enumerate(st) if s]
    return b, outs


def sweep_files(sub):
    files, gts = [], []
    for i, w in enumerate(WIDTHS):
        for j, h in enumerate(HEIGHTS):
            f, g = synth.synth_jpeg(20000 + 100 * i + j, w, h, sub, quality=[60, 85, 95][(i + j) % 3], want_coefs=True)
            files.append(f)
            gts.append(g)
    return files, gts


@pytest.mark.parametrize("sub", SUBS)
def test_shape_sweep_all_output_formats(sub):
    """136 shapes across the 128-px tiles of the IDCT/colour kernel (widths 1..641, heights 1..33) for each fused
    variant: once as one batch (>= 192 images with a second copy: the three-group path), in all three output
    formats, then in small batches; coefficients against the encoder's, every sample against ref64."""
    files, gts = sweep_files(sub)
    big = files + files[::-1]
    b, outs = decode(big)
    coefs = [b.coefficients(i) for i in range(len(big))]
    for i, g in enumerate(gts + gts[::-1]):
        for a, w in zip(coefs[i], g):
            assert np.array_equal(a[:len(w)], w[:len(a)]), i
    stats = ref64.Stats()
    check_images(big, coefs, outs, f"{sub} interleaved", stats)
    for fmt in (_ffi.OUT_RGB_PLANAR, _ffi.OUT_F32_PLANAR):
        b.set_output_format(fmt)
        if fmt == _ffi.OUT_F32_PLANAR:
            b.set_normalisation(SCALE, BIAS)
        b.idct()
        o2 = b.download()
        b.results()
        check_images(big, coefs, o2, f"{sub} format {fmt}", stats, fmt=fmt)
    b.close()
    for k in range(0, len(files), 8):
        part = files[k:k + 8]
        b, o3 = decode(part)
        c3 = [b.coefficients(i) for i in range(len(part))]
        b.close()
        for i in range(len(part)):
            assert all(np.array_equal(x, y) for x, y in zip(c3[i], coefs[k + i]))
        check_images(part, c3, o3, f"{sub} small batch {k}", stats)
    print(f"{sub}: {stats.samples} samples checked, {stats.band_fraction:.5f} in the band")


def test_compose_path_fancy_and_non_interleaved():
    """SPEC_FANCY (triangle filter) on interleaved files and files with one non-interleaved scan per component, box
    replication on the latter: every sample against ref64 in float64."""
    cases = [("420", 640, 480), ("422", 333, 217), ("440", 96, 160), ("420", 131, 77), ("444", 200, 100), ("420", 129, 9)]
    inter = [synth.synth_jpeg(21000 + i, w, h, s) for i, (s, w, h) in enumerate(cases)]
    b, outs = decode(inter, LAYOUT_SPEC_FANCY)
    coefs = [b.coefficients(i) for i in range(len(inter))]
    b.close()
    stats = ref64.Stats()
    check_images(inter, coefs, outs, "fancy", stats, fancy=True)
    planar = [synth.synth_jpeg(21000 + i, w, h, s, planar_scans=True) for i, (s, w, h) in enumerate(cases)]
    for layout in (LAYOUT_SPEC, LAYOUT_SPEC_FANCY):
        outs, st, cs = decode_scans(planar, ext=EXT_DRI, layout=layout, want_coefs=True)
        assert st == [0] * len(planar)
        for i, f in enumerate(planar):
            _, ds, _ = parse_scans(f, EXT_DRI, layout)
            fr = ref64.frame_from_descriptor(None, cs[i], fancy=layout == LAYOUT_SPEC_FANCY, scans=ds)   # one array per scan
            r = ref64.check_u8(fr, outs[i])
            assert r.bad == 0, (layout, i, r.first_bad)
    print(f"fancy interleaved: {stats.band_fraction:.5f} in the band")


def test_large_images_against_ref64():
    """The 16384 x 8192 4:2:0 image (134 Mpixel) and 3840 x 2160 4:4:4 images with and without restart intervals,
    where the oracle's O(N^4) IDCT is too slow: every sample against ref64, processed in row bands."""
    w, h = 16384, 8192
    f = synth.synth_jpeg(77, w, h, "420")
    k4 = [synth.synth_jpeg(3, 3840, 2160, "444", restart_interval=ri) for ri in (0, 16)]
    for files in ([f], k4):
        b, outs = decode(files)
        coefs = [b.coefficients(i) for i in range(len(files))]
        b.close()
        for i, fi in enumerate(files):
            t0 = time.time()
            st = ref64.check_u8(frame_of(fi, coefs[i]), outs[i], band_rows=256)
            assert st.bad == 0, (i, st.first_bad)
            print(f"{outs[i].shape}: {st.samples} samples, {st.band_fraction:.5f} in the band, ref64 check {time.time() - t0:.1f} s")


def test_randomised_batch_every_image():
    """The mixed random generator of test_randomised_batches (sampling, size, quality, restart interval): every image's
    pixels against ref64, coefficients against the encoder's."""
    rng = random.Random(4242)
    files, gts = [], []
    for it in range(120):
        sub = rng.choice(["420", "420", "422", "444", "440", "gray"])
        w = rng.choice([rng.randint(8, 300), rng.randint(300, 1400), rng.choice([512, 1024, 2048])])
        h = rng.choice([rng.randint(8, 300), rng.randint(300, 1000), rng.choice([512, 1024])])
        ri = rng.choice([0, 0, 1, 2, 3, 5, 8, 16, 33, 64, 100, 256, 1000])
        f, g = synth.synth_jpeg(rng.randint(0, 10 ** 6), w, h, sub, quality=rng.choice([30, 60, 85, 95]), restart_interval=ri, want_coefs=True)
        files.append(f)
        gts.append(g)
    b, outs = decode(files)
    coefs = [b.coefficients(i) for i in range(len(files))]
    b.close()
    for i in range(len(files)):
        for a, g in zip(coefs[i], gts[i]):
            assert np.array_equal(a[:len(g)], g[:len(a)]), i
    stats = ref64.Stats()
    check_images(files, coefs, outs, "random", stats)
    print(f"random batch: {stats.samples} samples, {stats.band_fraction:.5f} in the band")


CASES = craft.extreme_cases()


def check_crafted(cases):
    files = [c[1] for c in cases]
    b = Batch(files, layout=LAYOUT_SPEC, ext=EXT_DRI)
    b.upload().decode()
    outs = b.download()
    st, _ = b.results()
    for i, (name, f, want, dri) in enumerate(cases):
        o = O.decode(f, layout=O.LAYOUT_SPEC, ext=EXT_DRI if dri else EXT_NONE)
        assert st[i] == o.status == 0, (name, _ffi.status_string(st[i]), o.msg)
        got = b.coefficients(i)
        for a, w in zip(got, o.coefs):
            d = np.argwhere(a != w)
            assert not len(d), f"{name}: block {d[0][0]} position {d[0][1]}: {a[tuple(d[0])]} != {w[tuple(d[0])]}"
        r = ref64.check_u8(frame_of(f, got), outs[i])
        assert r.bad == 0, (name, r.first_bad)
    b.close()


def test_crafted_extremes():
    """All crafted files in one batch (distinct Huffman and quantisation tables per image): DC categories 12-16 with
    both leading bits, AC categories 11-15, overlong runs, ZRL at the end of a block, blocks without EOB, codes of
    every length with the canonical walk (second-level pool overflow, DC category 16 on a 2-bit code), single-basis
    blocks at +-1 / +-1023 / +-32767 with q = 1 / 255 / 65535, DC predictors past the int16 range, extremes only in
    chroma: coefficients bit-exact with the oracle, statuses equal, samples against ref64."""
    check_crafted(CASES)


@pytest.mark.parametrize("interval_mode,sync_multi", [("0", "0"), ("1", "0"), ("0", "1"), ("1", "1")])
def test_dc_walk_across_subsequences_and_intervals(interval_mode, sync_multi, monkeypatch):
    """The DC predictor walks (past +32767, back, past -32768) across 1024-bit subsequences and restart intervals,
    under both interval modes and both synchronisation passes, the write pass cut in two."""
    monkeypatch.setenv("JPGPU_SUBSEQ_BITS", "1024")
    monkeypatch.setenv("JPGPU_INTERVAL_MODE", interval_mode)
    monkeypatch.setenv("JPGPU_SYNC_MULTI", sync_multi)
    monkeypatch.setenv("JPGPU_WRITE_PARTS", "2")
    check_crafted([c for c in CASES if c[0].startswith(("dc_", "graded", "chroma"))])
