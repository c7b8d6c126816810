"""CPU build of the per-span walkers (akshar_b200/csrc/ak_text_core.cuh, compiled by g++ as a test aid) against the
oracle: cutting the buffer into arbitrary spans must never change the result -- the property the CUDA kernels rely on."""
import numpy as np
import pytest

import akshar_oracle as O
import oracle_batch as OB
import synth_corpus as sc
import walker_harness as W


import functools


@functools.lru_cache(None)
def _lines():
    lines = sc.adversarial(800, 21, 48) + sc.Corpus('social', 5).lines(8000) + sc.Corpus('hindi', 6).lines(5000)
    lines += ['', '', 'a', '', 'aaa', 'aa', '\n\n\n', '\u0958\u0958\u0958', 'e\u0301' * 5, '\u0928\u200c\u093c', '']
    return tuple(lines)


@functools.lru_cache(None)
def _exp_norm(flags):
    return OB.normalize_batch(_lines(), bool(flags & 1), bool(flags & 6))


@functools.lru_cache(None)
def _exp_seg(matras):
    return OB.segment_batch(_lines(), matras=matras)


@functools.lru_cache(None)
def _exp_runs():
    return OB.runs_batch(_lines())


@pytest.mark.parametrize('flags', [7, 6, 1, 0])
@pytest.mark.parametrize('span', [1, 3, 16, 64, 100000])
def test_normalize_spans(flags, span):
    lines = _lines()
    data, off = sc.pack(lines)
    exp, exp_off = _exp_norm(flags)
    out, out_off, st = W.normalize(data, off, flags=flags, span=span)
    assert st == 0
    assert np.array_equal(out_off, exp_off)
    assert out.tobytes() == exp.tobytes()


def test_normalize_random_spans():
    lines = _lines()
    data, off = sc.pack(lines)
    exp, exp_off = _exp_norm(7)
    rng = np.random.default_rng(3)
    for _ in range(3):
        out, out_off, st = W.normalize(data, off, flags=7, span=40, rng=rng)
        assert st == 0
        assert np.array_equal(out_off, exp_off)
        assert out.tobytes() == exp.tobytes()


@pytest.mark.parametrize('span', [1, 5, 32, 100000])
def test_segment_spans(span):
    lines = _lines()
    data, off = sc.pack(lines)
    ce, cs = _exp_seg(False)
    re_, rt, rs = _exp_runs()
    gce, gcs, gre, grt, grs, st = W.segment(data, off, flags=1 | 4, span=span)
    assert st == 0
    assert np.array_equal(gcs, cs) and np.array_equal(gce, ce)
    assert np.array_equal(grs, rs) and np.array_equal(gre, re_) and np.array_equal(grt, rt)
    me, ms = _exp_seg(True)
    gce, gcs, _, _, _, st = W.segment(data, off, flags=1 | 2, span=span)
    assert st == 0
    assert np.array_equal(gcs, ms) and np.array_equal(gce, me)


def test_bounded_lookback_flags_pathological():
    # a long run of Extend characters: a bounded backward walk must give up loudly, never answer wrongly
    lines = ['क' + 'ु' * 400 + 'ख']
    data, off = sc.pack(lines)
    _, _, _, _, _, st = W.segment(data, off, flags=1, span=16, limit=64)
    assert st & 4
    ce, cs = OB.segment_batch(lines)
    gce, gcs, _, _, _, st = W.segment(data, off, flags=1, span=16, limit=0)
    assert st == 0 and np.array_equal(gce, ce)


@pytest.mark.parametrize('flags,fn', [(1 | 8, O.semantic_normalize), (2 | 8, O.filter_garbage), (4 | 8, O.remove_elongations),
                                      (6 | 8, O.normalize_hinglish), (0, O.normalize_unicode)])
def test_single_stage_flags(flags, fn):
    lines = _lines()
    data, off = sc.pack(lines)
    exp = [fn(s).encode('utf-8') for s in lines]
    for span in (4, 32):
        out, out_off, st = W.normalize(data, off, flags=flags, span=span)
        assert st == 0
        b = out.tobytes()
        assert [b[out_off[i]:out_off[i + 1]] for i in range(len(lines))] == exp


# ---- bit-parallel normalize (ak_bits.cuh / ak_norm3.cuh): the kernel's lane phases and exchange rounds on the CPU
def test_basis_planes():
    rng = np.random.default_rng(1)
    for _ in range(100):
        b = rng.integers(0, 256, 32).astype(np.uint8)
        P = W.n3_planes(b)
        for k in range(8):
            assert int(P[k]) == sum(((int(b[i]) >> k) & 1) << i for i in range(32))


def test_byte_roles_match_the_tables():
    """the plane logic hard-codes byte classes; they must agree with the modules that own each rule"""
    import unicodedata as u
    import regex
    allowed = regex.compile(r'[\u0900-\u097F\u0980-\u09FFa-zA-Z0-9\s.,!?;:\'\"\-]')
    names = ['cont', 'K', 'NL', 'E0b', 'F0b', 'LXo', 'A4b', 'A5b', 'A6b', 'A7b', 'x9Fb', 'NKb', 'NIb', 'R2b', 'R3b', 'QNb', 'B6b',
             'B7b', 'low5']
    sets = {'A4b': {0xA4}, 'A5b': {0xA5}, 'A6b': {0xA6}, 'A7b': {0xA7}, 'x9Fb': {0x9F}, 'NKb': {0xBC}, 'R2b': {0x8D},
            'R3b': set(range(0x91, 0x95)), 'QNb': set(range(0x98, 0xA0)), 'NIb': {0xA8, 0xA9, 0xB0, 0xB1, 0xB3, 0xB4},
            'B6b': {0xBC, 0xBE}, 'B7b': {0x87, 0x8B, 0x8C, 0x8D, 0x97, 0x9C, 0x9D, 0x9F, 0xBE}, 'NL': {0x0A}, 'E0b': {0xE0},
            'F0b': {0xF0}, 'cont': set(range(0x80, 0xC0)), 'LXo': set(range(0xC0, 0x100)) - {0xE0, 0xF0}}
    for b in range(256):
        r = W.n3_roles(b)
        assert r != 0xFFFFFFFF
        g = lambda n: (r >> names.index(n)) & 1
        assert g('K') == (b < 0x80 and bool(allowed.match(chr(b))))
        for n, st in sets.items():
            assert g(n) == (b in st), (n, hex(b))
        low = (b | 0x20) if 0x41 <= b <= 0x5A else b
        assert g('low5') == ((low >> 5) & 1)
    # U+0900-09FF: the code points NFC can touch are exactly the ones the role masks single out
    for c in range(0x900, 0xA00):
        ch = chr(c)
        special = bool(u.combining(ch) or u.normalize('NFC', ch) != ch or u.decomposition(ch)
                       or c in (0x928, 0x930, 0x933, 0x9C7, 0x9BE, 0x9D7))
        b1, b2 = 0xA4 + ((c - 0x900) >> 6), 0x80 + (c & 63)
        if b1 == 0xA4:
            mine = b2 in sets['NKb'] | sets['NIb']
        elif b1 == 0xA5:
            mine = b2 in sets['R2b'] | sets['R3b'] | sets['QNb']
        elif b1 == 0xA6:
            mine = b2 in sets['B6b']
        else:
            mine = b2 in sets['B7b']
        assert special == mine, hex(c)
    # U+0928 / 0930 / 0933 are the bases a nukta composes with; 09C7 + 09BE / 09D7 likewise
    for a, m in ((0x928, 0x93C), (0x930, 0x93C), (0x933, 0x93C), (0x9C7, 0x9BE), (0x9C7, 0x9D7)):
        assert len(u.normalize('NFC', chr(a) + chr(m))) == 1
    # F0 9F xx xx (U+1F000-1FFFF) is dropped without a table look-up: plain for NFC, not allowed, no lower()
    for c in range(0x1F000, 0x20000):
        ch = chr(c)
        assert u.combining(ch) == 0 and u.normalize('NFC', 'a' + ch) == 'a' + ch and not allowed.match(ch)
        assert ch.lower() == ch


@pytest.mark.parametrize('real', [30, 1, 4])
def test_bit_parallel_lane_structure(real):
    lines = list(_lines())
    data, off = sc.pack(lines)
    exp, exp_off = _exp_norm(7)
    out, out_off, st, n_slow = W.fast_normalize3(data, off, real=real)
    assert st == 0
    assert np.array_equal(out_off, exp_off)
    assert out.tobytes() == exp.tobytes()


@pytest.mark.parametrize('real', [30, 3])
def test_bit_parallel_raw_mode(real):
    """normalize_text(clean_hinglish=False) through the same lanes: NFC + Roman lowercase, nothing dropped or collapsed"""
    lines = list(_lines()) + ['\u0130x', '\u00c9a', 'AAA\U0001F600aaa']
    data, off = sc.pack(lines)
    exp, exp_off = OB.normalize_batch(lines, True, False)
    out, out_off, st, n_slow = W.fast_normalize3(data, off, real=real, flags=1)
    assert st == 0
    assert np.array_equal(out_off, exp_off)
    assert out.tobytes() == exp.tobytes()
    for kind in ('hinglish', 'social'):
        lines = sc.Corpus(kind, 8).lines(100000)
        data, off = sc.pack(lines)
        exp, exp_off = OB.normalize_batch(lines, True, False)
        out, out_off, st, n_slow = W.fast_normalize3(data, off, real=real, flags=1)
        assert st == 0 and np.array_equal(out_off, exp_off) and out.tobytes() == exp.tobytes()
        assert n_slow / (data.size / 16) < 0.02


def test_bit_parallel_fuzz():
    """alphabets that keep most lanes fast: elongations across dropped stretches, row starts everywhere, rare trouble"""
    alpha = ['a', 'A', 'e', ' ', ' ', '\U0001F600', '\u0915', '\u093e', '\u094d', '\n', '!', '#', 'x', '\u0921', '\u0950',
             '\u0995', '_', '\t', '\U0001F468\u200d\U0001F469\u200d\U0001F467', 'a', 'a', ' ', '\u0915', '\u0915', '\u09bf', '\u09e6']
    tr = ['\u093c', '\u0928', '\u0951', 'e\u0301', '\u095c', '\u0130', '\u00a0', '\u00c9']
    rng = np.random.default_rng(5)
    for seed, (max_len, real) in enumerate([(120, 30), (40, 30), (300, 7), (8, 2), (64, 13)]):
        lines = sc.adversarial(1500, 500 + seed, max_len, alphabet=alpha)
        if seed >= 3:
            lines = [s if rng.random() < 0.7 else s[:len(s) // 2] + tr[int(rng.integers(len(tr)))] + s[len(s) // 2:] for s in lines]
        data, off = sc.pack(lines)
        exp, exp_off = OB.normalize_batch(lines)
        out, out_off, st, _ = W.fast_normalize3(data, off, real=real)
        assert st == 0 and np.array_equal(out_off, exp_off) and out.tobytes() == exp.tobytes()


def _zalgo_lines():
    import random
    rng = random.Random(11)
    marks = [chr(c) for c in (0x300, 0x301, 0x302, 0x303, 0x308, 0x30a, 0x316, 0x317, 0x323, 0x324, 0x325, 0x327, 0x328, 0x32d,
                              0x334, 0x335, 0x336, 0x338, 0x340, 0x341, 0x343, 0x344, 0x345, 0x35c, 0x360, 0x489, 0x93c, 0x94d,
                              0x951, 0x952)]
    excl = [chr(c) for c in range(0x958, 0x960)] + ['\ufb2a', '\ufb2b', '\ufb2e', '\ufb4b', '\u0f43', '\u2adc']
    lines = []
    for i in range(300):
        parts = []
        for _ in range(rng.choice((1, 3, 8))):
            base = rng.choice('aeou AEH\u0915\u0930\u0928z')
            k = rng.choice((0, 1, 5, 20, 45, 70, 120, 200, 240))
            parts.append(base + ''.join(rng.choice(marks) for _ in range(k)))
        lines.append(' '.join(parts))
    for i in range(200):
        n = rng.choice((1, 7, 40, 200, 700))
        lines.append(''.join(rng.choice('\u0915\u093e\u0964') if k % 20 == 19 else rng.choice(excl) for k in range(n)))
    return lines


def test_zalgo_and_expanding_text():
    """up to 240 stacked marks on one base (one NFC segment of up to 256 code points) and letters NFC makes longer:
    the walker alone (spans of 32 bytes) and the bit-parallel lanes with their slow-lane walker agree with the oracle;
    past the segment buffer the status says so"""
    lines = _zalgo_lines()
    data, off = sc.pack(lines)
    for flags, (nr, nc) in ((7, (True, True)), (1, (True, False))):
        exp, exp_off = OB.normalize_batch(lines, nr, nc)
        out, out_off, st = W.normalize(data, off, flags=flags, span=32)
        assert st == 0 and np.array_equal(out_off, exp_off) and out.tobytes() == exp.tobytes()
        out, out_off, st, _ = W.fast_normalize3(data, off, real=30, flags=flags)
        assert st == 0 and np.array_equal(out_off, exp_off) and out.tobytes() == exp.tobytes()
    data, off = sc.pack(['a' + '\u0301' * 300, '\u0958' * 200])
    assert W.normalize(data, off, flags=7, span=32)[2] & 2          # AKSHAR_ST_NFC_SEGMENT
    # akshars and script runs of the same text (normalized with nothing dropped, so the marks are still there)
    norm = [O.normalize_text(t, True, False) for t in lines]
    data, off = sc.pack(norm)
    ce, cs = OB.segment_batch(norm)
    re_, rt, rs = OB.runs_batch(norm)
    gce, gcs, gre, grt, grs, st = W.segment(data, off, flags=1 | 4, span=32)
    assert st == 0 and np.array_equal(gcs, cs) and np.array_equal(gce, ce)
    assert np.array_equal(grs, rs) and np.array_equal(gre, re_) and np.array_equal(grt, rt)


def wide_unicode_lines():
    """3000 strings drawn from 38 blocks (combining marks, Hebrew / Arabic, nine Indic scripts, Hangul jamo and syllables,
    compatibility ideographs, variation selectors, tags, flags, emoji ...)"""
    import random
    import unicodedata as u
    rng = random.Random(2026)
    blocks = [(0x20, 0x7f), (0xa0, 0x17f), (0x300, 0x36f), (0x370, 0x3ff), (0x590, 0x5ff), (0x600, 0x6ff), (0x900, 0x97f),
              (0x980, 0x9ff), (0xa00, 0xa7f), (0xb80, 0xbff), (0xc00, 0xc7f), (0xd00, 0xd7f), (0xe00, 0xe7f), (0xf00, 0xfff),
              (0x1000, 0x109f), (0x1100, 0x11ff), (0x1b00, 0x1b7f), (0x1e00, 0x1eff), (0x1f00, 0x1fff), (0x2000, 0x206f),
              (0x20d0, 0x20ff), (0x2190, 0x21ff), (0x2600, 0x27bf), (0x3040, 0x30ff), (0xa960, 0xa97f), (0xac00, 0xd7ff),
              (0xf900, 0xfaff), (0xfb00, 0xfb4f), (0xfe00, 0xfe0f), (0xfe20, 0xfe2f), (0x11000, 0x1107f), (0x11300, 0x1137f),
              (0x1d100, 0x1d1ff), (0x1f1e6, 0x1f1ff), (0x1f300, 0x1f6ff), (0x1f900, 0x1f9ff), (0xe0020, 0xe007f),
              (0xe0100, 0xe01ef)]

    def rcp():
        while True:
            a, b = rng.choice(blocks)
            c = rng.randint(a, b)
            if 0xd800 <= c <= 0xdfff or (u.category(chr(c)) == 'Cn' and rng.random() < 0.9):
                continue
            return chr(c)
    lines = []
    for i in range(3000):
        n = rng.choice((1, 2, 5, 12, 30, 80))
        pool = [rcp() for _ in range(rng.choice((2, 4, 8)))]
        s = ''.join(rng.choice(pool) if rng.random() < 0.6 else rcp() for _ in range(n))
        lines.append(s.replace('\n', ' ').replace('\r', ' '))
    return lines


def test_wide_unicode_fuzz(library_fuzz):
    """wide-Unicode strings: the oracle agrees with what the libraries the reference calls (unicodedata NFC, regex \\X)
    returned for them (recorded by tools/make_golden_fuzz.py), and walkers + bit-parallel lanes agree with the oracle"""
    lines = wide_unicode_lines()
    ref = library_fuzz['walkers']
    assert lines == ref['rows'], 'the generated rows are not the recorded ones'
    assert [O.normalize_unicode(s) for s in lines] == ref['nfc']
    assert [O.segment_akshars(s) for s in lines] == ref['clusters']
    data, off = sc.pack(lines)
    for flags, (nr, nc) in ((1, (True, False)), (7, (True, True)), (0, (False, False))):
        exp, exp_off = OB.normalize_batch(lines, nr, nc)
        out, out_off, st = W.normalize(data, off, flags=flags, span=32)
        assert st == 0 and np.array_equal(out_off, exp_off) and out.tobytes() == exp.tobytes()
        if flags:
            out, out_off, st, _ = W.fast_normalize3(data, off, real=30, flags=flags)
            assert st == 0 and np.array_equal(out_off, exp_off) and out.tobytes() == exp.tobytes()
    ce, cs = OB.segment_batch(lines)
    re_, rt, rs = OB.runs_batch(lines)
    for got in (W.segment(data, off, flags=1 | 4, span=32), W.seg_fast3(data, off, flags=1 | 4, real=30)):
        gce, gcs, gre, grt, grs, st = got[:6]
        assert st == 0 and np.array_equal(gcs, cs) and np.array_equal(gce, ce)
        assert np.array_equal(grs, rs) and np.array_equal(gre, re_) and np.array_equal(grt, rt)
    me, ms = OB.segment_batch(lines, matras=True)
    for got in (W.segment(data, off, flags=1 | 2, span=32), W.seg_fast3(data, off, flags=1 | 2, real=30)):
        assert got[5] == 0 and np.array_equal(got[1], ms) and np.array_equal(got[0], me)


def test_bit_parallel_is_mostly_fast():
    for kind in ('hinglish', 'hindi', 'social'):
        lines = sc.Corpus(kind, 8).lines(200000)
        data, off = sc.pack(lines)
        out, out_off, st, n_slow = W.fast_normalize3(data, off)
        exp, exp_off = OB.normalize_batch(lines)
        assert st == 0 and np.array_equal(out_off, exp_off) and out.tobytes() == exp.tobytes()
        assert n_slow / (data.size / 16) < 0.03


# ---- bit-parallel segmentation (ak_seg3.cuh)
def test_segment_byte_roles_match_the_tables():
    import json
    import os
    t = json.load(open(os.path.join(os.path.dirname(O.__file__), 'ucd_tables.json')))

    def expand(name):
        a = np.zeros(0x110000, dtype=np.int32)
        for r in t[name]:
            a[r[0]:r[1] + 1] = r[2]
        return a
    gcb, incb = expand('gcb'), expand('incb')
    names = ['cont', 'E0b', 'A4b', 'A5b', 'X4b', 'S4b', 'C4b', 'X5b', 'S5b', 'C5b', 'LKb', 'M4b', 'M5b', 'CR', 'LF', 'CTL', 'ROM', 'WEAK']
    is_matra = lambda c: 0x900 <= c <= 0x902 or 0x93E <= c <= 0x94D or 0x951 <= c <= 0x954        # segment.py:20-37
    for b in range(256):
        r = W.s3_roles(b)
        assert r != 0xFFFFFFFF
        g = lambda n: (r >> names.index(n)) & 1
        assert g('cont') == (0x80 <= b < 0xC0) and g('E0b') == (b == 0xE0) and g('A4b') == (b == 0xA4) and g('A5b') == (b == 0xA5)
        if 0x80 <= b < 0xC0:
            c4, c5 = 0x900 + (b & 63), 0x940 + (b & 63)
            assert g('X4b') == (gcb[c4] == 4) and g('S4b') == (gcb[c4] == 8) and g('C4b') == (incb[c4] == 1), hex(c4)
            assert g('X5b') == (gcb[c5] == 4) and g('S5b') == (gcb[c5] == 8) and g('C5b') == (incb[c5] == 1), hex(c5)
            assert g('LKb') == (incb[c5] == 2) and g('M4b') == is_matra(c4) and g('M5b') == is_matra(c5)
            for c in (c4, c5):      # what the fast lane assumes about the block
                assert gcb[c] in (0, 4, 8) and (incb[c] in (2, 3)) == (gcb[c] == 4)
        if b < 0x80:
            ch = chr(b)
            assert g('CR') == (b == 0x0D) and g('LF') == (b == 0x0A) and g('CTL') == (gcb[b] == 3)
            assert g('ROM') == (O.identify_script(ch) == 'roman')
            assert g('WEAK') == (O.identify_script(ch) in ('digit', 'punct')), ch


def _seg3_check(lines, real):
    data, off = sc.pack(lines)
    ce, cs = OB.segment_batch(lines)
    re_, rt, rs = OB.runs_batch(lines)
    gce, gcs, gre, grt, grs, st, ns = W.seg_fast3(data, off, flags=1 | 4, real=real)
    assert st == 0
    assert np.array_equal(gcs, cs) and np.array_equal(gce, ce)
    assert np.array_equal(grs, rs) and np.array_equal(gre, re_) and np.array_equal(grt, rt)
    me, ms = OB.segment_batch(lines, matras=True)
    gce, gcs, _, _, _, st, _ = W.seg_fast3(data, off, flags=1 | 2, real=real)
    assert st == 0
    assert np.array_equal(gcs, ms) and np.array_equal(gce, me)
    return ns / max(1.0, data.size / 32)


@pytest.mark.parametrize('real', [30, 1, 4])
def test_segment_bit_parallel_structure(real):
    _seg3_check(list(_lines()), real)


def test_segment_bit_parallel_fuzz():
    alpha = ['a', 'Z', 'e', ' ', ' ', '1', '9', '.', '-', '(', '\u0915', '\u093e', '\u094d', '\u094d', '\u093f', '\u0902', '\u093c',
             '\u0937', '\u0930', '\r', '\n', '\t', '\x01', '\x7f', '_', '@', '\u0950', '\u0964', '\u0966', '\u0962', '\u0903',
             '\u0904', '\u0915', '\u0915', '\u0921', '\u097b', '!', '[', '}']
    rng = np.random.default_rng(9)

    def rand_lines(n, max_len, alpha):
        out = []
        for _ in range(n):
            n_ch = int(rng.integers(0, max_len + 1))
            if rng.random() < 0.6:
                s = ''.join(alpha[int(i)] for i in rng.integers(0, len(alpha), size=n_ch))
            else:
                s = ''
                while len(s) < n_ch:
                    s += alpha[int(rng.integers(len(alpha)))] * int(rng.integers(1, 40))
            out.append(s)
        return out
    for max_len, real in [(120, 30), (400, 7), (6, 2)]:
        _seg3_check(rand_lines(1500, max_len, alpha), real)                                      # closed alphabet: fast lanes
        _seg3_check(rand_lines(800, max_len, alpha + ['\U0001F600', '\u0995', '\u200d', '\u00a0', 'e\u0301']), real)     # + foreign
    _seg3_check(['1234567890' * 20, '.' * 100 + 'a' + '.' * 70 + '\u0915', '\u094d' * 40 + '\u0915', '\u0915' + '\u094d' * 40 + '\u0915',
                 '\u0915\u094d' + '\u093c' * 30 + '\u0915', '\r\n' * 40, ''], 30)


def test_segment_bit_parallel_emoji_and_flags():
    """code points outside ASCII / U+0900-097F join the masks from the property table: GB11 (ZWJ sequences), GB12/13 (pairs
    of regional indicators, also across lanes), variation selectors, accents, other scripts; Hangul / Prepend take the walker"""
    rng = np.random.default_rng(4)
    alpha = ['\U0001F600', '\U0001F468', '\U0001F469', '\U0001F467', '\u200d', '\u200d', '\U0001F3FD', '\ufe0f', '\U0001F1EE',
             '\U0001F1F3', '\U0001F1FA', '\U0001F1F8', '\u2764', '\u2728', 'a', ' ', '\u0915', '\u094d', '\u0937', '\u00e9', '\u0301',
             '\u200b', '\u00ad', '1', '.', '\u00a9', '\u20e3', '#', '\U0001F3F3', '\U0001F308', '\n', '\r', '\u200c', '\u0995',
             '\u09cd', '\u09b7', '\u0966', '\u0663']

    def rand_lines(n, max_len, alpha):
        out = []
        for _ in range(n):
            n_ch = int(rng.integers(0, max_len + 1))
            if rng.random() < 0.5:
                s = ''.join(alpha[int(i)] for i in rng.integers(0, len(alpha), size=n_ch))
            else:
                s = ''
                while len(s) < n_ch:
                    s += alpha[int(rng.integers(len(alpha)))] * int(rng.integers(1, 12))
            out.append(s)
        return out
    for max_len, real in [(60, 30), (200, 7), (12, 2)]:
        assert _seg3_check(rand_lines(1500, max_len, alpha), real) < 0.10
        _seg3_check(rand_lines(500, max_len, alpha + ['\uac00', '\u1100', '\u1161', '\u0600']), real)          # + unsupported classes
    raw = sc.Corpus('social', 8).lines(100000)
    assert _seg3_check(raw, 30) < 0.001                  # emoji, ZWJ families, flags, accents: all in the fast lanes


def test_segment_bit_parallel_is_all_fast_on_normalized_text():
    for kind in ('hinglish', 'hindi', 'social'):
        lines = [O.normalize_text(s) for s in sc.Corpus(kind, 8).lines(100000)]
        assert _seg3_check(lines, 30) < 0.001


# ---- word tokenizers (ak_wordtok.cuh; reference segment.py:239-401) -------------------------------------------------
def _words_expected(lines, mode):
    """token (begin, end) byte offsets per row from the oracle's loops over the text AS IT IS (normalizing is the caller's job)"""
    loop = O._word_loop if mode == 0 else O._split_loop
    begin, end, splits, flags = [], [], [0], []
    for s in lines:
        cps = [ord(c) for c in s]
        pre = [0]
        for cp in cps:
            pre.append(pre[-1] + O.utf8_len(cp))
        for b, e in loop(cps):
            begin.append(pre[b])
            end.append(pre[e])
        splits.append(len(begin))
        flags.append(1 if any(0x0900 <= cp <= 0x097F for cp in cps) else 0)
    return np.array(begin, dtype=np.int32), np.array(end, dtype=np.int32), np.array(splits, dtype=np.int64), np.array(flags, dtype=np.uint8)


def _words_check(lines, real):
    data, off = sc.pack(lines)
    for mode in (0, 1):
        eb, ee, es, ef = _words_expected(lines, mode)
        wb, we, sp, fl, st = W.wordtok(data, off, mode=mode, real=real)
        assert st == 0
        assert np.array_equal(sp, es)
        assert np.array_equal(wb, eb) and np.array_equal(we, ee)
        assert np.array_equal(fl, ef)


@pytest.mark.parametrize('real', [30, 1, 5])
def test_word_tokenizer_lane_structure(real):
    lines = list(_lines())
    _words_check(lines, real)                                           # raw text: every kind of character
    _words_check([O.normalize_text(s) for s in lines[:3000]], real)     # what word_tokenize_hindi feeds the loop


def test_word_tokenizer_fuzz():
    alpha = ['a', 'Z', ' ', ' ', '1', '.', ',', '!', '?', ';', ':', '(', ')', '[', ']', '{', '}', '"', "'", '-', '_', 'क', 'ा',
             '्', '।', '॥', '।', '॰', '\t', '\n', '\x0b', '\x0c', '\r', '\x1c', '\x1d', '\x1e', '\x1f', '\x00',
             '\x7f', '\x85', '\xa0', ' ', ' ', ' ', '​', ' ', ' ', ' ', ' ', '　',
             '、', '\U0001F600', 'ক', '\xe9', 'ॣ', '०', '@', '/', '\\']
    rng = np.random.default_rng(12)
    for max_len, real in [(150, 30), (500, 3), (5, 2), (40, 30)]:
        lines = []
        for _ in range(1500):
            n_ch = int(rng.integers(0, max_len + 1))
            if rng.random() < 0.7:
                lines.append(''.join(alpha[int(i)] for i in rng.integers(0, len(alpha), size=n_ch)))
            else:
                s = ''
                while len(s) < n_ch:
                    s += alpha[int(rng.integers(len(alpha)))] * int(rng.integers(1, 70))
                lines.append(s)
        _words_check(lines, real)
    _words_check(['', '', '।', '', 'a' * 200, '', ' ' * 100, '॥' * 50, 'a।', '।a', ''], 30)
    _words_check(['क' * 31 + '।', 'ab' + '।' * 10 + 'c', 'x' * 29 + '।' + 'y'], 30)           # danda across lanes


# ---- file bytes -> rows (ak_lines.cuh; reference cli.py:165-190) -----------------------------------------------------
def test_file_rows_like_readlines_and_strip(tmp_path):
    rng = np.random.default_rng(3)
    alpha = ['a', 'b', ' ', ' ', '\n', '\n', '\r', '\r\n', '\t', '\x0b', '\x0c', '\x1c', '\x1d', '\x1e', '\x1f', '\x85', '\xa0', '\u1680',
             '\u2000', '\u200a', '\u200b', '\u2028', '\u2029', '\u202f', '\u205f', '\u3000', '\u0915', '\u093e', '\U0001F600', '\ufeff', 'x y']
    for trial in range(60):
        n = int(rng.integers(0, 400))
        if trial % 3 == 0:
            s = ''.join(alpha[int(i)] for i in rng.integers(0, len(alpha), size=n))
        else:
            s = ''
            while len(s) < n:
                s += alpha[int(rng.integers(len(alpha)))] * int(rng.integers(1, 50))
        data = s.encode('utf-8')
        exp = O.file_rows(data)
        # the restatement against Python's own text-mode file
        p = tmp_path / 'f.txt'
        p.write_bytes(data)
        with open(p, 'r', encoding='utf-8') as f:
            assert [ln.strip() for ln in f.readlines() if ln.strip()] == exp
        for span in (32, 1, 5, 1000):
            assert [r.decode('utf-8') for r in W.lines(data, span=span)] == exp
        for lead in (0, 7, 15):                                       # the kernels' lanes: bit masks per 32 bytes
            assert [r.decode('utf-8') for r in W.lines32(data, lead=lead)] == exp
    for s in ('', '\n', 'a', 'a\n', '\na', ' a ', '\r\r\n\r', 'a\rb\r\nc\n\nd', ' ' * 100 + 'a' + ' ' * 100, '\u3000\u0915\u3000', 'a' * 100):
        assert [r.decode('utf-8') for r in W.lines(s.encode('utf-8'))] == O.file_rows(s.encode('utf-8'))
        assert [r.decode('utf-8') for r in W.lines32(s.encode('utf-8'))] == O.file_rows(s.encode('utf-8'))
