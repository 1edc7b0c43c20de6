"""Scans on which the look-back synchronisation of the entropy stage cannot fall into step, so that the repair rounds of
verify_scan_kernel (and of the CPU simulation) do the work.  Test infrastructure, built on craft.write_jpeg.

Every generator returns (file bytes, per component the reference's coefficients).  Two ambiguities drive them:

* zigzag phase (gray): every symbol is four bits and means the same thing as a DC and as an AC symbol, and the long
  blocks have no EOB.  A decoder that starts cold inside a block keeps its wrong zigzag index for good.
* MCU phase (colour): the luma DC code plus its one raw bit has the same bits as the chroma DC code, and all
  components share one AC table.  A decoder that starts on the wrong block of an MCU parses every block right and
  labels every one of them wrongly, for good.

A wrong phase must also change the coefficients, or a failed repair would go unnoticed (a flat image decodes the same
in every phase): each generator checks with a small bit-level decoder (`_decode`) that every wrong phase of its
adversarial stretch yields other coefficients than the true one.

The tables carry codes for every other baseline symbol too (all starting with bits the adversarial stretches never
use at a symbol start), so ordinary coefficients (`synth`) can surround an adversarial stretch in one scan."""
import numpy as np

import craft
from jpeg_rust_b200 import synth

SAMPLING = {"420": (2, 2), "422": (2, 1), "440": (1, 2), "444": (1, 1)}
_OTHER_AC = [s for s in craft.BASELINE_AC if s not in (0x00, 0x01, 0x02)]


def gray_tables():
    """DC "00" = category 2; AC "00" = run 0 / size 2, "01" = EOB; every other symbol on longer codes."""
    dc = craft.Table.from_lengths([(2, 2)] + [(s, 6) for s in range(12) if s != 2])
    ac = craft.Table.from_lengths([(0x02, 2), (0x00, 2), (0x01, 10)] + [(s, 10) for s in _OTHER_AC])
    return dc, ac


def colour_tables():
    """Luma DC "00" = category 1, so "00" + raw bit 1 reads "001"; chroma DC "001" = category 0; one AC table for
    all components: "00" = EOB, "01" = run 0 / size 1."""
    dcy = craft.Table.from_lengths([(1, 2)] + [(s, 6) for s in range(12) if s != 1])
    dcc = craft.Table.from_lengths([(2, 3), (0, 3)] + [(s, 6) for s in range(12) if s not in (0, 2)])
    ac = craft.Table.from_lengths([(0x00, 2), (0x01, 2), (0x02, 10)] + [(s, 10) for s in _OTHER_AC])
    assert dcy.code[1] == (0b00, 2) and dcc.code[0] == (0b001, 3)
    return dcy, dcc, ac


# ---------------------------------------------------------------------------------------------------------------------
# layout helpers: blocks are handled in decode order (MCU by MCU) as (component, symbol list)

def _layout(sub):
    """Per MCU position the component; the frame's component tuples for write_jpeg."""
    if sub == "gray":
        return [0], [(1, 1, 0, 0, 0)]
    h, v = SAMPLING[sub]
    return [0] * (h * v) + [1, 2], [(h, v, 0, 0, 0), (1, 1, 0, 1, 0), (1, 1, 0, 1, 0)]


def _mcus(sub, w, h):
    if sub == "gray":
        return -(-w // 8) * -(-h // 8)
    hh, vv = SAMPLING[sub]
    return -(-w // (8 * hh)) * -(-h // (8 * vv))


def _tables(sub):
    if sub == "gray":
        dc, ac = gray_tables()
        return [dc], [ac], {0: dc}, {0: ac}
    dcy, dcc, ac = colour_tables()
    return [dcy, dcc, dcc], [ac, ac, ac], {0: dcy, 1: dcc}, {0: ac}


def _symbols(labels, blocks):
    """Coefficient blocks (absolute DC) to symbol lists, with the DC predictors of the decode order."""
    pred = [0, 0, 0]
    out = []
    for i, b in enumerate(blocks):
        comp = labels[i % len(labels)]
        syms = b if isinstance(b, list) else craft.block_symbols(b, pred[comp])
        _, pred[comp] = craft.reference_block(syms, pred[comp])
        out.append(syms)
    return out


def _bit_length(syms, dc, ac):
    n = 0
    for k, (s, _) in enumerate(syms):
        n += (dc if k == 0 else ac).code[s][1] + (s if k == 0 else s & 15)
    return n


def _write(sub, w, h, blocks, ri=0):
    """blocks: symbol lists in decode order.  Returns write_jpeg's (file, coefficients per component)."""
    labels, comps = _layout(sub)
    _, _, dcs, acs = _tables(sub)
    per = [[] for _ in comps]
    for i, b in enumerate(blocks):
        per[labels[i % len(labels)]].append(b)
    return craft.write_jpeg(w, h, comps, per, {0: [1] * 64}, dcs, acs, ri)


def _flat(sub, want):
    """The reference's coefficients in decode order."""
    labels, _ = _layout(sub)
    nb = len(labels)
    taken = [0, 0, 0]
    out = []
    for i in range(sum(len(c) for c in want)):
        comp = labels[i % nb]
        out.append(want[comp][taken[comp]])
        taken[comp] += 1
    return out


# ---------------------------------------------------------------------------------------------------------------------
# the phase check

def _bits_of(blocks, sub):
    """The entropy-coded bits of symbol lists (no restart markers, no stuffing), as a uint8 array of 0/1."""
    labels, _ = _layout(sub)
    dcs, acs, _, _ = _tables(sub)
    out = []
    for i, syms in enumerate(blocks):
        comp = labels[i % len(labels)]
        for k, (s, raw) in enumerate(syms):
            code, ln = (dcs if k == 0 else acs)[comp].code[s]
            out.append(format(code, f"0{ln}b"))
            size = s if k == 0 else s & 15
            if size:
                out.append(format(raw, f"0{size}b"))
    return np.frombuffer("".join(out).encode(), np.uint8) - ord("0")


def _decode(bits, p, sub, c, z, pred, nblocks):
    """The reference's block decode (craft.reference_block) from bit p with the decoder believing it is at block c of
    an MCU, zigzag index z: nblocks blocks (zigzag, absolute DC), or None where a code is not in its table."""
    labels, _ = _layout(sub)
    dcs, acs, _, _ = _tables(sub)
    inv = {}

    def table(t):
        if id(t) not in inv:
            inv[id(t)] = {(ln, code): s for s, (code, ln) in t.code.items()}
        return inv[id(t)]

    def read(n):
        nonlocal p
        v = 0
        for _ in range(n):
            v = (v << 1) | int(bits[p]) if p < len(bits) else (v << 1) | 1
            p += 1
        return v

    def symbol(t):
        m, code = table(t), 0
        for ln in range(1, 17):
            code = (code << 1) | read(1)
            if (ln, code) in m:
                return m[(ln, code)]
        return None

    pred = list(pred)
    out = []
    for _ in range(nblocks):
        comp = labels[c]
        blk = [0] * 64
        if z == 0:
            s = symbol(dcs[comp])
            if s is None:
                return None
            pred[comp] += craft.value_correction(read(s), s)
            blk[0] = max(-32768, min(32767, pred[comp]))
            z = 1
        while z < 64:
            s = symbol(acs[comp])
            if s is None:
                return None
            if s == 0x00:
                break
            if s == 0xf0:
                z += 16
                continue
            z = min(z + (s >> 4), 63)
            blk[z] = craft.value_correction(read(s & 15), s & 15)
            z += 1
        out.append(np.array(blk, np.int16))
        c, z = (c + 1) % len(labels), 0
    return out


def check_wrong_phases_visible(sub, blocks, want, first, count=3):
    """Decodes `count` MCUs (gray: blocks) from the start of MCU `first` in the true phase and in every wrong one
    (gray: zigzag index 1..63 at a block start; colour: every other block of the MCU).  The true phase must reproduce
    the reference's coefficients and every wrong phase must differ from them in a block it decoded whole."""
    labels, _ = _layout(sub)
    nb = len(labels)
    dcs, acs, _, _ = _tables(sub)
    bits = _bits_of(blocks, sub)
    flat = _flat(sub, want)
    b0 = first * nb
    p = sum(_bit_length(blocks[i], dcs[labels[i % nb]], acs[labels[i % nb]]) for i in range(b0))
    pred = [0, 0, 0]
    for i in range(b0):
        pred[labels[i % nb]] = int(flat[i][0])
    n = count * nb
    truth = _decode(bits, p, sub, 0, 0, pred, n)
    assert all(np.array_equal(a, e) for a, e in zip(truth, flat[b0:b0 + n])), "the bit-level decoder disagrees"
    phases = [(0, z) for z in range(1, 64)] if sub == "gray" else [(c, 0) for c in range(1, nb)]
    for c, z in phases:
        got = _decode(bits, p, sub, c, z, pred, n + 1)
        if got is None:
            continue
        whole = got[1:] if z else got          # a decoder starting at z > 0 completes a partial block first
        assert any(not np.array_equal(a, e) for a, e in zip(whole, flat[b0 + (1 if z else 0):])), \
            f"{sub}: the wrong phase (block {c}, zigzag {z}) decodes to the same coefficients"


# ---------------------------------------------------------------------------------------------------------------------
# the generators

def _chain_blocks(n, lead):
    """Gray zigzag-phase chain: two short blocks (DC + `lead` AC symbols + EOB, DC + EOB: 3 + lead nibbles), then
    blocks of 64 four-bit symbols without EOB, DC +3 / -3 alternately ("0011" / "0000"), AC +3 ("0011").  The long
    blocks sit 3 + lead nibbles off the 256-bit grid, so every cold start at a multiple of 256 bits takes nibble
    64 - (3 + lead) % 64 of a block for a DC symbol and keeps that zigzag phase: A(j) == B(j-1) holds for every link but
    the first, and each repair round mends exactly one link (nsub - 1 rounds)."""
    assert 0 <= lead <= 62 and (3 + lead) % 64 != 0
    out = [[(2, 3)] + [(0x02, 3)] * lead + [(0x00, 0)], [(2, 0), (0x00, 0)]]
    for b in range(2, n):
        out.append([(2, 3 if b % 2 == 0 else 0)] + [(0x02, 3)] * 63)
    return out


def _crowd_block(comp, rng):
    """An MCU-phase block: DC "001" (luma +1, chroma 0), 0-3 AC values +-1 at run 0, EOB."""
    return [(1, 1) if comp == 0 else (0, 0)] + [(0x01, int(rng.integers(0, 2))) for _ in range(int(rng.integers(0, 4)))] + [(0x00, 0)]


def _crowd_blocks(sub, nmcu, rng):
    """MCU-phase content of random length: cold starts land on every block of the MCU, many links break at once and
    stay broken until the correct prefix reaches them (a repair from a wrong predecessor keeps its wrong phase)."""
    labels, _ = _layout(sub)
    return [_crowd_block(labels[i % len(labels)], rng) for i in range(nmcu * len(labels))]


def _chain_colour_blocks(sub, nmcu):
    """MCU-phase chain for MCUs of four blocks (4:2:2, 4:4:0): every block "001" + "01 1" + "00" (8 bits, MCU 32 bits),
    but the first has 8 more AC values (24 bits): the MCUs sit 24 bits off the 256-bit grid, and every cold start
    begins on block 1 of an MCU believing it block 0."""
    labels, _ = _layout(sub)
    assert len(labels) == 4
    out = [[(1, 1) if labels[i % 4] == 0 else (0, 0), (0x01, 1), (0x00, 0)] for i in range(nmcu * 4)]
    out[0] = [(1, 1)] + [(0x01, 1)] * 9 + [(0x00, 0)]
    return out


def zigzag_chain(w, h, lead=0, ri=0):
    """(a) w x h gray, see _chain_blocks; `lead` moves the wrong zigzag phase.  ri: restart interval in blocks."""
    blocks = _chain_blocks(_mcus("gray", w, h), lead)
    f, want = _write("gray", w, h, blocks, ri)
    if ri == 0:
        check_wrong_phases_visible("gray", blocks, want, 2)
    return f, want


def mcu_phase(sub, w, h, seed=0, ri=0):
    """(b) MCU-phase ambiguity, 4:2:0 / 4:2:2 / 4:4:0 / 4:4:4, see _crowd_blocks."""
    blocks = _crowd_blocks(sub, _mcus(sub, w, h), np.random.default_rng(seed))
    f, want = _write(sub, w, h, blocks, ri)
    if ri == 0:
        check_wrong_phases_visible(sub, blocks, want, 5)
    return f, want


def chain_then_crowd(sub, w, h, chain_fraction=0.5, seed=0, ri=0):
    """(c) the MCU-phase chain of _chain_colour_blocks over the first part of the scan, then MCU-phase content of
    random length: the chain is mended one link per round, its link the lowest broken one, while the crowd above it
    keeps more than kRepairJobs (256) links broken in the early rounds (at 1024-bit subsequences and full size: up to
    450-630 of them, in the first 220-400 rounds); after that the crowd's count falls below 256 and the chain's last
    part is mended alone."""
    n = _mcus(sub, w, h)
    k = int(n * chain_fraction)
    blocks = _chain_colour_blocks(sub, k) + _crowd_blocks(sub, n - k, np.random.default_rng(seed))
    f, want = _write(sub, w, h, blocks, ri)
    if ri == 0:
        check_wrong_phases_visible(sub, blocks, want, 3)
        check_wrong_phases_visible(sub, blocks, want, k + 3)
    return f, want


def stitched(kind, sub, w, h, seed=0):
    """(e) the coefficients of a synth image, with the MCUs of its middle third replaced by an adversarial stretch
    (kind "chain": the gray zigzag chain, lead-in included; "crowd": MCU-phase content): the repairs must leave no
    trace in the ordinary coefficients after the stretch."""
    _, coefs = synth.synth_jpeg(seed, w, h, sub, want_coefs=True)
    labels, _ = _layout(sub)
    nb = len(labels)
    n = _mcus(sub, w, h)
    taken = [0, 0, 0]
    ordinary = []
    for i in range(n * nb):
        c = labels[i % nb]
        ordinary.append(np.asarray(coefs[c][taken[c]], np.int64))
        taken[c] += 1
    lo, hi = n // 3, 2 * n // 3
    if kind == "chain":
        assert sub == "gray"
        middle = _chain_blocks(hi - lo, 5)
    else:
        middle = _crowd_blocks(sub, hi - lo, np.random.default_rng(seed))
    blocks = _symbols(labels, ordinary[:lo * nb] + middle + ordinary[hi * nb:])
    f, want = _write(sub, w, h, blocks)
    check_wrong_phases_visible(sub, blocks, want, lo + 4)
    flat = _flat(sub, want)
    for i in list(range(lo * nb)) + list(range(hi * nb, n * nb)):   # the ordinary parts keep their values (DC aside)
        assert np.array_equal(flat[i][1:], ordinary[i][1:]), i
    return f, want


class Case:
    def __init__(self, name, kind, f, want, ri=0):
        self.name, self.kind, self.file, self.want, self.ri = name, kind, f, want, ri


def corpus(small=False):
    """The adversarial corpus.  Full size: nsub >= 1024 at 1024-bit subsequences for the chains and the crowds (more
    than 256 broken links in a round); small: the same constructions at a quarter of the area.  Restart intervals:
    the gray chain's blocks are 256 bits, so 12 blocks are exactly three 1024-bit subsequences (13 are not); the
    crowd's intervals are some 3.6 subsequences, long enough for the synchronisation pass to run."""
    d = 2 if small else 1
    cases = [Case("chain_lead0", "chain", *zigzag_chain(512 // d, 512, lead=0)),
             Case("chain_lead17", "chain", *zigzag_chain(256, 512 // d, lead=17)),
             Case("chain_lead40", "chain", *zigzag_chain(512 // d, 256, lead=40))]
    for i, (sub, w, h) in enumerate([("420", 2560, 2048), ("422", 2048, 2048), ("440", 2048, 2048), ("444", 2048, 1280)]):
        cases.append(Case(f"crowd_{sub}", "crowd", *mcu_phase(sub, w // d, h // d, seed=i)))
    cases.append(Case("chain_then_crowd_422", "chain_crowd", *chain_then_crowd("422", 2048 // d, 2048 // d, seed=7)))
    cases.append(Case("chain_then_crowd_440", "chain_crowd", *chain_then_crowd("440", 2048 // d, 2048 // d, 0.3, seed=8)))
    for ri in (12, 13):
        cases.append(Case(f"chain_dri{ri}", "chain_dri", *zigzag_chain(512 // d, 256, lead=0, ri=ri), ri=ri))
    cases.append(Case("crowd_420_dri64", "crowd_dri", *mcu_phase("420", 1024 // d, 1024, seed=9, ri=64), ri=64))
    cases.append(Case("stitched_chain_gray", "stitched", *stitched("chain", "gray", 640, 480, seed=10)))
    cases.append(Case("stitched_crowd_420", "stitched", *stitched("crowd", "420", 640, 480, seed=11)))
    cases.append(Case("stitched_crowd_444", "stitched", *stitched("crowd", "444", 496, 368, seed=12)))
    return cases


# Planner settings (environment) as a pairwise-covering array: 16 rows, every pair of values of any two switches in
# some row.  Row (i, k): subsequence bits i, (sync, verify multi-symbol) k; the others follow from i and k.
# The pairs are pairs of requested values; some collapse in the planner: write-pass units are capped by the
# subsequence length (1 at 1024 bits, at most 2 at 2048: jpgpu_host.cpp, never shorter than 1024 bits), a checkpoint
# distance of 512 bits is already the default up to 4096-bit subsequences, and JPGPU_VERIFY_MULTI=1 has no effect
# when JPGPU_SYNC_MULTI=0 (the repair walks use the multi-symbol tables only when the synchronisation pass loads
# them).  Over the effective values, besides the pairs the planner rules out, these pairs are not met: 4 write-pass
# units with no look-back; the default checkpoint distances of 8192- and 32768-bit subsequences (1024 and 4096 bits)
# with the planner's look-back; 1024-bit checkpoints with one write-pass unit; 4096-bit checkpoints with 4 units and
# with the multi-symbol repair walks.
_SUB = ["1024", "2048", "8192", "32768"]
_LOOKBACK = ["0", None, "8192"]          # None: the planner's choice
_SEG = ["512", None]
_PARTS = ["1", "2", "4"]


def settings():
    rows = []
    for i in range(4):
        for k in range(4):
            rows.append({"JPGPU_SUBSEQ_BITS": _SUB[i], "JPGPU_SYNC_MULTI": str(k >> 1), "JPGPU_VERIFY_MULTI": str(k & 1),
                         "JPGPU_LOOKBACK_BITS": _LOOKBACK[(i + k) % 3], "JPGPU_SEG_BITS": _SEG[(i + k) % 2],
                         "JPGPU_WRITE_PARTS": _PARTS[(i + 2 * k) % 3], "JPGPU_INTERVAL_MODE": str((i + k // 2) % 2)})
    return rows


def settings_id(row):
    return "-".join(f"{k[6:].lower()}{v}" for k, v in row.items() if v is not None)


def apply(monkeypatch, row):
    for k, v in row.items():
        if v is None:
            monkeypatch.delenv(k, raising=False)
        else:
            monkeypatch.setenv(k, v)


def entropy_data(f):
    """The bytes between the SOS header and the closing EOI of a file written by craft.write_jpeg (stuffing and
    restart markers included)."""
    i = 2
    while True:
        assert f[i] == 0xff
        m, n = f[i + 1], (f[i + 2] << 8) | f[i + 3]
        i += 2 + n
        if m == 0xda:
            break
    assert f[-2:] == b"\xff\xd9"
    return f[i:len(f) - 2]


def scan_bits(f):
    """Bits of the entropy-coded data after unstuffing and without restart markers (what the subsequences cut)."""
    data = entropy_data(f)
    out, k = 0, 0
    while k < len(data):
        if data[k] == 0xff:
            k += 2          # stuffed 0x00 or a marker: the 0xff byte stays only when stuffed
            out += 1 if data[k - 1] == 0x00 else 0
            continue
        out += 1
        k += 1
    return out * 8


def nsub(f, sub_bits):
    return -(-scan_bits(f) // sub_bits)
