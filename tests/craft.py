"""Entropy writer for chosen coefficients or symbol sequences: baseline JPEG files whose scans hold exactly what a test
asks for, including what the in-repo encoder never produces (DC size categories 12-16, AC categories 11-15, DC
predictors past the int16 range, codes of every length 2-16, runs past position 63, ZRL at the end of a block, blocks
without an EOB).  Test infrastructure.

A block is either 64 zigzag coefficients with an absolute DC (coded the usual way: DC difference against the
component's predictor, run/size symbols, ZRL, EOB) or a list of symbols (sym, raw): `sym` the Huffman symbol (the size
category for the block's first, DC, symbol; run << 4 | size, 0x00 EOB, 0xf0 ZRL after it) and `raw` its `size` value
bits as written.  Along with the file the writer returns the coefficients the reference makes of it (decoder.rs:195-215,
huffman.rs:146-195, 256-268): DC differences and values through value_correction in i16 (category 16 = the raw bits
read as an i16), the DC predictor summed unsaturated and stored `as i16` (saturating)."""
import numpy as np

ZIGZAG = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6,
                   7, 14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31,
                   39, 46, 53, 60, 61, 54, 47, 55, 62, 63])   # zigzag position -> natural (row * 8 + col) index


class Table:
    """A Huffman table as DHT carries it: bits[l - 1] codes of length l, then the symbols in code order."""

    def __init__(self, bits, vals):
        assert len(bits) == 16 and sum(bits) == len(vals) <= 256
        self.bits, self.vals = [int(b) for b in bits], [int(v) for v in vals]
        self.code = {}                               # symbol -> (code, length): T.81 C.2
        code, k = 0, 0
        for ln in range(1, 17):
            for _ in range(self.bits[ln - 1]):
                assert code < (1 << ln), "not a prefix code"
                self.code[self.vals[k]] = (code, ln)
                code += 1
                k += 1
            code <<= 1
        assert all(c != (1 << ln) - 1 for c, ln in self.code.values()), "an all-ones code collides with the fill bits"

    @staticmethod
    def from_lengths(lengths):
        """lengths: list of (symbol, code length) in the order the codes are to be handed out within a length."""
        bits = [0] * 16
        for _, ln in lengths:
            bits[ln - 1] += 1
        vals = [s for s, _ in sorted(lengths, key=lambda sl: sl[1])]   # stable: keeps the order within a length
        return Table(bits, vals)


def graded_table(symbols, first_len=2):
    """One code of each length first_len..15 for the first symbols, every further symbol at length 16: a table with
    codes of every length (T.81 caps a DHT at 256 symbols)."""
    out = []
    for i, s in enumerate(symbols):
        out.append((s, min(first_len + i, 16)))
    return Table.from_lengths(out)


BASELINE_AC = [0x00, 0xf0] + [(r << 4) | s for r in range(16) for s in range(1, 11)]   # the 162 symbols of T.81 K.3
EXTENDED_AC = BASELINE_AC + [(r << 4) | s for r in range(16) for s in range(11, 16)]  # + categories 11-15: 242 symbols


def default_tables():
    """DC categories 0-16 and every AC symbol (242), short codes for the common symbols."""
    dc = Table.from_lengths([(s, 5) for s in range(0, 16)] + [(16, 6)])
    ac_common = [0x00, 0x01, 0x11, 0x02, 0xf0]
    rest = [s for s in EXTENDED_AC if s not in ac_common]
    ac = Table.from_lengths([(s, 3) for s in ac_common] + [(s, 9) for s in rest[:100]] + [(s, 12) for s in rest[100:]])
    return dc, ac


def value_bits(v):
    """T.81 F.1.2.1: size category and the raw bits of a value."""
    s = int(abs(int(v))).bit_length()
    return s, (int(v) if v >= 0 else int(v) + (1 << s) - 1)


def value_correction(raw, size):
    """huffman.rs:256-268 in i16: T.81 EXTEND for size <= 15; size 16 reads the raw bits as an i16."""
    if size == 0:
        return 0
    if size == 16:
        return raw - 65536 if raw & 0x8000 else raw
    return raw if raw >> (size - 1) else raw - (1 << size) + 1


def block_symbols(zz, pred):
    """Symbols of a block of 64 zigzag coefficients (absolute DC) against the predictor `pred`."""
    zz = [int(x) for x in zz]
    diff = zz[0] - pred
    if not -32767 <= diff <= 32767:
        raise ValueError(f"DC difference {diff} has no size category <= 15")
    s, raw = value_bits(diff)
    out, run = [(s, raw)], 0
    for k in range(1, 64):
        if zz[k] == 0:
            run += 1
            continue
        if not -32767 <= zz[k] <= 32767:
            raise ValueError(f"AC value {zz[k]} has no size category <= 15")
        while run > 15:
            out.append((0xf0, 0))
            run -= 16
        s, raw = value_bits(zz[k])
        out.append(((run << 4) | s, raw))
        run = 0
    if run:
        out.append((0x00, 0))
    return out


def reference_block(syms, pred):
    """huffman.rs:146-195 + decoder.rs:208-210 on a symbol list: (zigzag block, new predictor).  The list must end
    with the symbol that completes the block."""
    s, raw = syms[0]
    pred += value_correction(raw, s)
    blk = [max(-32768, min(32767, pred))]
    k = 1
    while len(blk) < 64:
        assert k < len(syms), "the symbols end before the block"
        sym, raw = syms[k]
        k += 1
        if sym == 0x00:
            blk += [0] * (64 - len(blk))
        elif sym == 0xf0:
            blk += [0] * min(16, 64 - len(blk))
        else:
            blk += [0] * min(sym >> 4, 64 - len(blk) - 1)
            blk.append(value_correction(raw, sym & 15))
    assert k == len(syms), "symbols after the end of the block"
    return blk, pred


class BitWriter:
    def __init__(self):
        self.out, self.acc, self.n = bytearray(), 0, 0

    def put(self, value, nbits):
        assert 0 <= value < (1 << nbits) or nbits == 0
        self.acc = (self.acc << nbits) | value
        self.n += nbits
        while self.n >= 8:
            self.n -= 8
            byte = (self.acc >> self.n) & 0xff
            self.out.append(byte)
            if byte == 0xff:
                self.out.append(0x00)                        # byte stuffing (T.81 F.1.2.3)
        self.acc &= (1 << self.n) - 1

    def flush_ones(self):
        if self.n:
            self.put((1 << (8 - self.n)) - 1, 8 - self.n)    # 1-padding to the byte boundary


def _segment(marker, payload):
    n = len(payload) + 2
    return bytes([0xff, marker, n >> 8, n & 0xff]) + bytes(payload)


def dqt(tid, values, wide=None):
    """A DQT segment: 64 values in zigzag order, 8-bit entries unless a value needs 16 bits (or wide=True)."""
    values = [int(v) for v in values]
    assert len(values) == 64 and all(1 <= v <= 65535 for v in values)
    wide = max(values) > 255 if wide is None else wide
    p = [(0x10 if wide else 0) | tid]
    for v in values:
        p += [v >> 8, v & 0xff] if wide else [v]
    return _segment(0xdb, p)


def write_jpeg(width, height, comps, blocks, qts, dc_tables, ac_tables, restart_interval=0, wide_dqt=None):
    """comps: list of (h, v, tq, td, ta) per component; blocks: per component its blocks in MCU order (T.81 A.2.3:
    MCU by MCU, the component's v rows of h blocks each), coefficient arrays or symbol lists; qts: {tq: 64 zigzag
    values}; dc_tables / ac_tables: {id: Table}.  Returns (file bytes, per component the reference's (n, 64) int16
    coefficients)."""
    hmax, vmax = max(c[0] for c in comps), max(c[1] for c in comps)
    if len(comps) == 1:
        mcux, mcuy = -(-width // 8), -(-height // 8)
        per = [1]
    else:
        mcux, mcuy = -(-width // (8 * hmax)), -(-height // (8 * vmax))
        per = [h * v for h, v, _, _, _ in comps]
    nmcu = mcux * mcuy
    for c, b in enumerate(blocks):
        assert len(b) == nmcu * per[c], f"component {c}: {len(b)} blocks for {nmcu} MCUs of {per[c]}"
    o = bytearray([0xff, 0xd8])
    for tid, q in sorted(qts.items()):
        o += dqt(tid, q, wide_dqt)
    p = [8, height >> 8, height & 0xff, width >> 8, width & 0xff, len(comps)]
    for i, (h, v, tq, _, _) in enumerate(comps):
        p += [i + 1, (h << 4) | v, tq]
    o += _segment(0xc0, p)
    for tc, tabs in ((0, dc_tables), (1, ac_tables)):
        for tid, t in sorted(tabs.items()):
            o += _segment(0xc4, [(tc << 4) | tid] + t.bits + t.vals)
    if restart_interval:
        o += _segment(0xdd, [restart_interval >> 8, restart_interval & 0xff])
    p = [len(comps)]
    for i, (_, _, _, td, ta) in enumerate(comps):
        p += [i + 1, (td << 4) | ta]
    o += _segment(0xda, p + [0, 63, 0])
    bw = BitWriter()
    expect = [[] for _ in comps]
    pred, written = [0] * len(comps), [0] * len(comps)
    rst = 0
    for m in range(nmcu):
        if restart_interval and m and m % restart_interval == 0:
            bw.flush_ones()
            bw.out += bytes([0xff, 0xd0 + (rst & 7)])
            rst += 1
            pred = [0] * len(comps)
        for c, (_, _, _, td, ta) in enumerate(comps):
            for _ in range(per[c]):
                b = blocks[c][written[c]]
                written[c] += 1
                syms = b if isinstance(b, list) and (not b or isinstance(b[0], tuple)) else block_symbols(b, pred[c])
                blk, pred[c] = reference_block(syms, pred[c])
                expect[c].append(blk)
                for k, (sym, raw) in enumerate(syms):
                    code, ln = (dc_tables[td] if k == 0 else ac_tables[ta]).code[sym]
                    bw.put(code, ln)
                    size = sym if k == 0 else sym & 15
                    if size:
                        bw.put(raw, size)
    bw.flush_ones()
    o += bw.out + bytes([0xff, 0xd9])
    return bytes(o), [np.array(e, np.int16).reshape(-1, 64) for e in expect]


def single_basis(k, value, dc=0):
    """A zigzag block with `value` at zigzag position k (and the DC `dc` when k > 0)."""
    zz = np.zeros(64, np.int64)
    zz[0] = dc
    zz[k] = value
    return zz


# ---- build_huff_lut's two levels (jpgpu_host.cpp), restated to tell which codes only the canonical walk decodes
LUT_BITS, POOL_SIZE = 9, 256


def canonical_walk_symbols(table, is_dc):
    """Symbols build_huff_lut leaves to the canonical walk: codes longer than kLutBits whose kLutBits-prefix got no
    second-level sub-table (the pool, kPoolSize entries, is handed out in prefix order) or that are longer than the
    sub-table is wide; for DC tables also size categories >= 16."""
    codes = [(c, ln, s) for s, (c, ln) in table.code.items() if not (is_dc and s >= 16)]
    maxlen = {}
    for c, ln, _ in codes:
        if ln > LUT_BITS:
            pre = c >> (ln - LUT_BITS)
            maxlen[pre] = max(maxlen.get(pre, 0), ln)
    used, width = 0, {}
    for pre in sorted(maxlen):
        nb = min(maxlen[pre] - LUT_BITS, 7)
        if used + (1 << nb) > POOL_SIZE:
            continue
        width[pre] = nb
        used += 1 << nb
    slow = {s for c, ln, s in codes if ln > LUT_BITS and (c >> (ln - LUT_BITS) not in width or ln > LUT_BITS + width[c >> (ln - LUT_BITS)])}
    if is_dc:
        slow |= {s for s in table.code if s >= 16}
    return slow


# ---------------------------------------------------------------------------------------------------------------------
# The crafted extremes both suites decode (test_reference64.py on the oracle and the CPU simulation,
# test_gpu_reference64.py on the device).  Each case: (name, file bytes, the reference's coefficients, uses DRI).

def _grid(nblocks, per_row=64):
    rows = -(-nblocks // per_row)
    return 8 * min(nblocks, per_row), 8 * rows, rows * min(nblocks, per_row)


def _gray(blocks, qt, dc, ac, ri=0, per_row=64, wide=None):
    w, h, n = _grid(len(blocks), per_row)
    assert n == len(blocks), (n, len(blocks))
    return write_jpeg(w, h, [(1, 1, 0, 0, 0)], [blocks], {0: qt}, {0: dc}, {0: ac}, ri, wide)


def single_basis_file(q):
    """Every zigzag position at +-1, +-1023, +-32767 with every quantisation entry q (16-bit DQT for q > 255): samples
    saturate both ways; DC offsets put the small ones across 0 and 255."""
    dc, ac = default_tables()
    base = {1: [0, -1020, 1012], 255: [0, -4, 4]}.get(q, [0, 0, 0])
    blocks = []
    for i, v in enumerate([1, -1, 1023, -1023, 32767, -32767]):
        for k in range(64):
            d = 0 if k in (0, 1, 63) else base[(i + k) % 3]   # DC differences stay within category 15
            blocks.append(single_basis(k, v, d) if k else single_basis(0, v))
    return _gray(blocks, [q] * 64, dc, ac)


def dc_walk_blocks(n_up=20, step=2047, rounds=3, rng=None):
    """DC differences walking the predictor up past +32767, staying there, down past -32768 and back, with a few AC
    values per block so the scan spans many 1024-bit subsequences.  Symbol lists: after a restart the same
    differences walk from 0 again."""
    rng = rng or np.random.default_rng(5)
    diffs = []
    for _ in range(rounds):
        for seg, s in ((n_up, step), (12, 0), (2 * n_up + 3, -step), (12, 0), (n_up, step)):
            diffs += [s] * seg
    blocks = []
    for d in diffs:
        zz = np.zeros(64, np.int64)
        zz[0] = d
        zz[rng.choice(np.arange(1, 64), 4, replace=False)] = rng.choice([-1023, -200, 37, 900], 4)
        blocks.append(block_symbols(zz, 0))
    return blocks


def dc_walk_file(ri=0):
    dc, ac = default_tables()
    blocks = dc_walk_blocks()
    return _gray(blocks[:len(blocks) // 16 * 16], [1] * 64, dc, ac, ri, per_row=16)


def issue_tables():
    """Small tables: DC 00 -> 0, 01 -> 11, 100 -> 15, 101 -> 16; AC 00 -> EOB."""
    return (Table.from_lengths([(0, 2), (11, 2), (15, 3), (16, 3)]), Table.from_lengths([(0x00, 2)]))


def dc_saturation_file():
    """20 blocks of DC difference +2047: the predictor passes 32767 at the 17th, the stored DC stays there."""
    dc, ac = issue_tables()
    return _gray([[(11, 2047), (0x00, 0)] for _ in range(20)], [1] * 64, dc, ac, per_row=20)


def dc_category16_file():
    """DC category 16 with both leading bits and at the extremes, through a 3-bit code."""
    dc, ac = issue_tables()
    raws = [0x0001, 0xffff, 0x8000, 0x7fff, 0x0000, 0x8001, 0x1234, 0xedcb]
    return _gray([[(16, r), (0x00, 0)] for r in raws], [1] * 64, dc, ac, per_row=8)


def _advance(z):
    """AC symbols taking a block from zigzag index 1 to z (values +-1; ZRLs while more than 16 zeros are left)."""
    out, blen = [], 1
    while z - blen > 16:
        out.append((0xf0, 0))
        blen += 16
    if z > blen:
        out.append((((z - blen - 1) << 4) | 1, 1))
    return out


def categories_and_runs_file():
    """DC categories 12-16 and AC categories 11-15 with both leading bits; runs that step past 63 from z = 49..62;
    ZRL reaching and passing 64; a block ending at 63 without an EOB; ZRL followed directly by EOB."""
    dc, ac = default_tables()
    blocks = []
    for s in range(12, 17):
        for raw in (1 << (s - 1), (1 << (s - 1)) - 1, (1 << s) - 1, 0):     # leading 1 / leading 0, both ends
            blocks.append([(s, raw), (0x00, 0)])
    for s in range(11, 16):
        for raw in (1 << (s - 1), (1 << (s - 1)) - 1, (1 << s) - 1, 0):
            blocks.append([(0, 0), (s, raw), ((15 << 4) | s, raw), (0x00, 0)])
    for z in range(49, 63):                                   # (run 15, size 1) from z: the value lands at 63
        blocks.append([(0, 0)] + _advance(z) + [(0xf1, 1)])
        blocks.append([(0, 0)] + _advance(z) + [((((63 - z) if z < 63 else 0) << 4) | 1, 0)])
    for z in (48, 50, 60, 63):                                # ZRL reaching / passing 64
        blocks.append([(0, 0)] + _advance(z) + [(0xf0, 0)])
    blocks.append([(0, 0)] + _advance(63) + [(0x01, 1)])      # coefficient 63, no EOB
    blocks.append([(0, 0)] + _advance(10) + [(0xf0, 0), (0x00, 0)])
    blocks.append([(0, 0), (0xf0, 0), (0xf0, 0), (0xf0, 0), (0x00, 0)])
    while len(blocks) % 16:
        blocks.append([(0, 0), (0x00, 0)])
    return _gray(blocks, [3] * 64, dc, ac, per_row=16)


def every_symbol_blocks(dc_syms, ac_syms, rng):
    """Blocks that use every DC and every AC symbol at least once (raw bits random, both leading bits)."""
    blocks, acs, k = [], list(ac_syms), 0
    dcs = [s for s in dc_syms]
    i = 0
    while k < len(acs) or i < len(dcs):
        s = dcs[i % len(dcs)]
        i += 1
        syms, blen = [(s, int(rng.integers(0, 1 << s)) if s else 0)], 1
        while k < len(acs):
            a = acs[k]
            if a == 0x00:
                k += 1
                continue
            adv = 16 if a == 0xf0 else (a >> 4) + 1
            if blen + adv > 63:
                break
            syms.append((a, int(rng.integers(0, 1 << (a & 15))) if a & 15 else 0))
            blen += adv
            k += 1
        syms.append((0x00, 0))
        blocks.append(syms)
    return blocks


def graded_tables_file(reverse, seed):
    """Codes of every length 2-16 in both tables; the AC table holds all 162 baseline symbols and categories 11-15
    (242), so its 16-bit codes overflow the second-level pool.  reverse: the rare symbols get the short codes (DC 16
    a 2-bit code)."""
    dc_order = list(range(17))[::-1] if reverse else list(range(17))
    ac_order = EXTENDED_AC[::-1] if reverse else EXTENDED_AC
    dc, ac = graded_table(dc_order), graded_table(ac_order)
    rng = np.random.default_rng(seed)
    blocks = every_symbol_blocks(dc_order, ac_order, rng)
    while len(blocks) % 16:
        blocks.append([(0, 0), (0x00, 0)])
    return _gray(blocks, [2] * 64, dc, ac, per_row=16), (dc, ac)


def chroma_extremes_file():
    """4:2:0: ordinary luma, every extreme in chroma (single-basis +-32767 with 16-bit quantisation, a DC walk past
    the int16 range)."""
    dc, ac = default_tables()
    rng = np.random.default_rng(11)
    mcux, mcuy = 8, 4
    n = mcux * mcuy
    y = []
    for _ in range(4 * n):
        zz = np.zeros(64, np.int64)
        zz[0] = int(rng.integers(-60, 60))
        zz[1:6] = rng.integers(-20, 20, 5)
        y.append(zz)
    cb = [single_basis(int(k % 63) + 1, 32767 if k % 2 else -32767) for k in range(n)]
    walk = dc_walk_blocks(n_up=4, step=9000, rounds=1)
    cr = [walk[k % len(walk)] for k in range(n)]
    return write_jpeg(16 * mcux, 16 * mcuy, [(2, 2, 0, 0, 0), (1, 1, 1, 1, 1), (1, 1, 1, 1, 1)], [y, cb, cr],
                      {0: [4] * 64, 1: [65535] * 64}, {0: dc, 1: dc}, {0: ac, 1: ac})


def extreme_cases():
    cases = []
    for q in (1, 255, 65535):
        cases.append((f"single_basis_q{q}", *single_basis_file(q), False))
    cases.append(("dc_saturation", *dc_saturation_file(), False))
    cases.append(("dc_category16", *dc_category16_file(), False))
    cases.append(("categories_and_runs", *categories_and_runs_file(), False))
    for rev in (False, True):
        (f, want), _ = graded_tables_file(rev, 21 + rev)
        cases.append((f"graded_tables{'_reversed' if rev else ''}", f, want, False))
    cases.append(("chroma_extremes_420", *chroma_extremes_file(), False))
    cases.append(("dc_walk", *dc_walk_file(0), False))
    cases.append(("dc_walk_dri", *dc_walk_file(37), True))
    return cases
