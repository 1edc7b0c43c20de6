"""The float64 reference of the IDCT / colour stage (ref64.py) pinned against the oracle, the crafted-file writer
(craft.py) against the oracle, and the crafted extremes on the CPU simulation (the same per-thread decode code as the
kernels): coefficients bit-exact, statuses equal, samples under ref64's rule."""
import numpy as np
import pytest

import craft
import oracle_ffi as O
import ref64
import sim_ffi as S
from conftest import fixture_bytes
from jpeg_rust_b200 import EXT_DRI, EXT_NONE, LAYOUT_SPEC, parse_descriptor, synth


def frame_of(data, coefs, ext=EXT_NONE):
    st, d, _ = parse_descriptor(data, ext, LAYOUT_SPEC)
    assert st == 0
    return ref64.frame_from_descriptor(d, coefs)


def test_ref64_against_the_oracle():
    """ref64 and the oracle's pixels agree under the rule with the oracle's float32 bound, on the fixtures and on
    synthetic images of all five sampling modes at ragged sizes and several qualities."""
    files = [fixture_bytes(n) for n in ("lena.jpeg", "lena-bw.jpeg", "2x2-chroma.jpeg")]
    for i, (s, w, h, q) in enumerate([("420", 333, 200, 85), ("422", 250, 131, 95), ("440", 129, 77, 50), ("444", 17, 9, 100),
                                      ("gray", 255, 33, 85), ("420", 1, 1, 30), ("440", 130, 257, 98), ("422", 641, 17, 5)]):
        files.append(synth.synth_jpeg(8300 + i, w, h, s, quality=q))
    for i, f in enumerate(files):
        o = O.decode(f, layout=O.LAYOUT_SPEC)
        assert o.status == 0
        st = ref64.check_u8(frame_of(f, o.coefs), o.rgb, c=ref64.C_ORACLE)
        print(f"file {i}: {st.samples} samples, {st.band_fraction:.5f} in the band")
        assert st.bad == 0, (i, st.bad, st.first_bad)


def test_ref64_catches_a_wrong_colour_constant():
    """The rule is tight enough to see 1.402 -> 1.4025 in the red channel, which the +-1 gate passes."""
    f = synth.synth_jpeg(8400, 256, 128, "444", quality=95)
    o = O.decode(f, layout=O.LAYOUT_SPEC)
    fr = frame_of(f, o.coefs)
    y, cr = o.planes[0] + np.float32(128.0), o.planes[2]
    bad = o.rgb.copy()
    bad[..., 0] = np.clip(np.trunc(cr * np.float32(1.4025) + y), 0, 255).astype(np.uint8)
    assert np.abs(bad.astype(int) - o.rgb.astype(int)).max() <= 1
    assert ref64.check_u8(fr, bad, c=ref64.C_ORACLE).bad > 0


def test_crafted_files_decode_to_the_intended_coefficients():
    """Every crafted file decodes on the oracle to what the writer meant, under the reference's semantics (i16
    value_correction, unsaturated f32 predictor stored saturated)."""
    for name, f, want, dri in craft.extreme_cases():
        o = O.decode(f, layout=O.LAYOUT_SPEC, ext=EXT_DRI if dri else EXT_NONE)
        assert o.status == 0, (name, o.msg)
        assert len(o.coefs) == len(want)
        for a, w in zip(o.coefs, want):
            assert np.array_equal(a, w), name


def test_crafted_writer_features():
    """Byte stuffing, RST markers in sequence with 1-padding, 16-bit DQT, and the tables the extremes rely on: codes
    of every length 2-16; an AC table with every baseline symbol whose long codes overflow the second-level pool."""
    f, _ = craft.dc_walk_file(37)
    scan = f[f.index(b"\xff\xda") + 10:-2]
    markers = [scan[i + 1] for i in range(len(scan) - 1) if scan[i] == 0xff and scan[i + 1] != 0]
    assert markers == [0xd0 + k % 8 for k in range(len(markers))] and len(markers) >= 8
    assert all(scan[i + 1] == 0 or 0xd0 <= scan[i + 1] <= 0xd7 for i in range(len(scan) - 1) if scan[i] == 0xff)
    f, _ = craft.single_basis_file(65535)
    assert b"\xff\xdb\x00\x83\x10" in f                       # Pq = 1, 128 bytes of entries
    (_, _), (dc, ac) = craft.graded_tables_file(False, 21)
    assert {ln for _, ln in dc.code.values()} == set(range(2, 17)) == {ln for _, ln in ac.code.values()}
    assert set(craft.BASELINE_AC) <= set(ac.code) and len(ac.code) == 242
    slow = craft.canonical_walk_symbols(ac, is_dc=False)
    assert slow and slow <= set(ac.code)
    assert craft.canonical_walk_symbols(dc, is_dc=True) == {16}


CASES = craft.extreme_cases()


def sim_check(cases, sub_bits=0):
    files = [c[1] for c in cases]
    rs, _ = S.decode_batch(files, layout=LAYOUT_SPEC, ext=EXT_DRI, sub_bits=sub_bits)
    for (name, f, want, dri), r in zip(cases, rs):
        o = O.decode(f, layout=O.LAYOUT_SPEC, ext=EXT_DRI if dri else EXT_NONE)
        assert r.status == o.status == 0, (name, r.status, o.msg)
        for a, w in zip(r.coefs, o.coefs):
            d = np.argwhere(a != w)
            assert not len(d), f"{name}: block {d[0][0]} position {d[0][1]}: {a[tuple(d[0])]} != {w[tuple(d[0])]}"
        st = ref64.check_u8(frame_of(f, r.coefs, EXT_DRI), r.rgb)
        assert st.bad == 0, (name, st.first_bad)


def test_crafted_extremes_on_the_simulation():
    """All crafted files in one simulated batch: DC categories 12-16 with both leading bits, AC categories 11-15,
    overlong runs, ZRL at the end of a block, blocks without EOB, codes of every length (canonical walk included),
    single-basis blocks at +-32767 with q up to 65535, DC predictors past the int16 range, extremes only in chroma."""
    sim_check(CASES)


@pytest.mark.parametrize("interval_mode,sync_multi", [("0", 0), ("1", 0), ("0", 1), ("1", 1)])
def test_dc_walk_across_subsequences_and_intervals(interval_mode, sync_multi, monkeypatch):
    """The DC predictor walk over 1024-bit subsequences (the synchronisation pass carries the unsaturated sums) and
    over restart intervals, in both interval modes, with and without the multi-symbol synchronisation tables, and
    with the write pass cut in two."""
    monkeypatch.setenv("JPGPU_INTERVAL_MODE", interval_mode)
    monkeypatch.setenv("JPGPU_WRITE_PARTS", "2")
    walks = [c for c in CASES if c[0].startswith("dc_") or c[0].startswith("graded") or c[0].startswith("chroma")]
    S.set_sync_multi(sync_multi)
    try:
        sim_check(walks, sub_bits=1024)
    finally:
        S.set_sync_multi(1)
