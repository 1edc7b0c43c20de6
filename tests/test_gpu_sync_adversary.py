"""The entropy stage on the device against scans that never self-synchronise (sync_adversary.py): serial chains of
broken links, crowds of more than 256 broken links per repair round, both at once, restart intervals, adversarial
stretches inside ordinary content.  Every image: status 0, coefficients bit-exact with the generator's (which the CPU
suite shows equal to the oracle's), bytes_read against the oracle without DRI, every sample under ref64."""
import functools
import random
import time

import numpy as np
import pytest

import oracle_ffi as O
import ref64
import sync_adversary as A
from jpeg_rust_b200 import EXT_DRI, LAYOUT_SPEC, Batch, _ffi, parse_descriptor, synth

pytestmark = pytest.mark.gpu

_ROWS = A.settings()


@functools.lru_cache(maxsize=None)
def _corpus():
    return A.corpus(False)


@functools.lru_cache(maxsize=None)
def _oracle_bytes_read(i):
    c = _corpus()[i]
    return O.decode(c.file, layout=O.LAYOUT_SPEC).bytes_read


_checked = {}   # image name -> samples that passed ref64 (a later decode of the same coefficients must equal them)


def _decode(files):
    b = Batch(files, layout=LAYOUT_SPEC, ext=EXT_DRI)
    b.upload().decode()
    outs = b.download()
    st, br = b.results()
    coefs = [b.coefficients(i) for i in range(len(files))]
    b.close()
    return st, br, coefs, outs


def _check(names, files, wants, st, coefs, outs):
    for i, (name, f, want) in enumerate(zip(names, files, wants)):
        assert st[i] == 0, (name, _ffi.status_string(st[i]))
        assert len(coefs[i]) == len(want), name
        for k, (a, w) in enumerate(zip(coefs[i], want)):
            if name.startswith("synth_"):    # the encoder's coefficients: the blocks of the image proper
                a, w = a[:len(w)], w[:len(a)]
            assert a.shape == w.shape, (name, k, a.shape, w.shape)
            d = np.argwhere(a != w)
            assert not len(d), f"{name} component {k}: block {d[0][0]} position {d[0][1]}: {a[tuple(d[0])]} != {w[tuple(d[0])]}"
        if name in _checked:
            assert np.array_equal(outs[i], _checked[name]), name
            continue
        _, desc, _ = parse_descriptor(f, EXT_DRI, LAYOUT_SPEC)
        r = ref64.check_u8(ref64.frame_from_descriptor(desc, coefs[i]), outs[i])
        assert r.bad == 0, (name, r.first_bad)
        _checked[name] = outs[i]


def _check_corpus(st, br, coefs, outs, idx):
    cases = _corpus()
    _check([cases[i].name for i in idx], [cases[i].file for i in idx], [cases[i].want for i in idx], st, coefs, outs)
    for k, i in enumerate(idx):
        if not cases[i].ri:
            assert br[k] == _oracle_bytes_read(i), (cases[i].name, br[k], _oracle_bytes_read(i))


@pytest.mark.parametrize("row", _ROWS, ids=A.settings_id)
def test_corpus_under_planner_settings(row, monkeypatch):
    """The whole corpus as one batch under each row of the pairwise-covering settings array (subsequence bits,
    look-back, checkpoint distance, write-pass units, single / multi-symbol synchronisation and repair walks, interval
    mode of the DRI files)."""
    A.apply(monkeypatch, row)
    idx = list(range(len(_corpus())))
    st, br, coefs, outs = _decode([c.file for c in _corpus()])
    _check_corpus(st, br, coefs, outs, idx)


def test_single_images_and_a_batch_of_eight():
    """Each adversarial image alone (one CTA repairs while the rest of the machine idles), then eight of them."""
    cases = _corpus()
    for i in range(len(cases)):
        st, br, coefs, outs = _decode([cases[i].file])
        _check_corpus(st, br, coefs, outs, [i])
    idx = [0, 3, 4, 7, 8, 9, 11, 13]
    st, br, coefs, outs = _decode([cases[i].file for i in idx])
    _check_corpus(st, br, coefs, outs, idx)


def _synth_files(n, seed):
    rng = random.Random(seed)
    out = []
    for k in range(n):
        sub = rng.choice(["420", "422", "444", "440", "gray"])
        f, g = synth.synth_jpeg(30000 + seed + k, rng.choice([64, 200, 320]), rng.choice([48, 144, 240]), sub,
                                restart_interval=rng.choice([0, 0, 0, 7]), want_coefs=True)
        out.append((f"synth_{seed}_{k}", f, g))
    return out


def _mixed(n_synth, seed, idx):
    cases = _corpus()
    items = [(cases[i].name, cases[i].file, cases[i].want) for i in idx] + _synth_files(n_synth, seed)
    random.Random(seed).shuffle(items)
    return items


def test_mixed_batch_three_groups_and_determinism():
    """The corpus among 190 synth images (>= 192: three image groups and the auxiliary streams, as the benchmark
    runs), decoded three times and once in reverse order: every output and every coefficient byte-identical (the
    repair work is handed out through atomics and barriers; its result must not depend on their timing)."""
    from jpeg_rust_b200 import plan_info
    items = _mixed(190, 1, range(len(_corpus())))
    names, files, wants = zip(*items)
    assert len(files) >= 192
    runs = [_decode(list(files)) for _ in range(3)]
    rev = _decode(list(files[::-1]))
    st, br, coefs, outs = runs[0]
    _check(names, files, wants, st, coefs, outs)
    for s2, b2, c2, o2 in runs[1:] + [tuple(x[::-1] for x in rev)]:
        assert s2 == st and b2 == br
        for i in range(len(files)):
            assert np.array_equal(o2[i], outs[i]), names[i]
            assert all(np.array_equal(x, y) for x, y in zip(c2[i], coefs[i])), names[i]
    assert plan_info(list(files), ext=EXT_DRI, layout=LAYOUT_SPEC)["groups"] == 3


def test_batch_past_444_images():
    """More than 444 images: the planner turns the multi-symbol repair walks off (the symbol-by-symbol walks of
    verify_scan_kernel<false> repair the corpus)."""
    items = _mixed(440, 2, range(len(_corpus())))
    names, files, wants = zip(*items)
    assert len(files) > 444
    st, br, coefs, outs = _decode(list(files))
    _check(names, files, wants, st, coefs, outs)


def test_time_of_the_longest_serial_chain(capsys):
    """2048 x 2048 gray zigzag chain at the planner's subsequence length: one CTA repairs about nsub links one after
    the other.  Reported, not asserted."""
    from jpeg_rust_b200 import plan_info
    f, want = A.zigzag_chain(2048, 2048, lead=0)
    sub_bits = plan_info([f], ext=EXT_DRI, layout=LAYOUT_SPEC)["sub_bits"]
    _decode([synth.synth_jpeg(1, 64, 64, "gray")])          # modules loaded, tables cached
    b = Batch([f], layout=LAYOUT_SPEC, ext=EXT_DRI)
    b.upload()
    b.ctx.sync()
    t0 = time.perf_counter()
    b.decode()
    b.ctx.sync()
    ms = (time.perf_counter() - t0) * 1e3
    outs = b.download()
    st, _ = b.results()
    coefs = [b.coefficients(0)]
    b.close()
    _check(["chain_2048"], [f], [want], st, coefs, outs)
    import torch
    dev = torch.cuda.get_device_name(0)
    with capsys.disabled():
        print(f"\n2048x2048 gray zigzag chain: scan {A.scan_bits(f)} bits, nsub {A.nsub(f, sub_bits)} at {sub_bits} "
              f"bits (the planner's choice), decode {ms:.1f} ms on {dev}")
