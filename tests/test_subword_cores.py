"""CPU build of the model loaders (ak_models.cpp) and subword cores (ak_subword.cuh, signature in ak_text_core.cuh)
against the vectors recorded from the unmodified reference (tests/golden) and the oracle.  Test aid only: the
product runs these same functions inside the CUDA kernels."""
import os

import numpy as np
import pytest

import akshar_oracle as O
import synth_corpus as sc
import walker_harness as W


def _rows(golden, limit=None):
    rows = golden['rows'] if limit is None else golden['rows'][:limit]
    return rows


def _walker_rows(rows):
    """the span walker (ak_bpe_span) on its own takes text HF's NFKC leaves alone; anything else goes through the row path
    of the event-stream encoder (test_bpe_event_stream, test_raw_mode_cores)"""
    T = O.tables()
    return [r for r in rows if all(T.bpe_safe[ord(c)] for c in r['norm'])]


@pytest.mark.parametrize('name', ['bpe24k', 'bpe_corpus'])
@pytest.mark.parametrize('span', [32, 7, 100000])
def test_bpe_ids_match_reference(golden, bpe_rows, models_dir, name, span):
    assert W.load_bpe(os.path.join(models_dir, name + '.json')) == golden['vocab_size'][name]
    rows = _walker_rows(bpe_rows)
    data, off = sc.pack([r['norm'] for r in rows])
    ids, splits, st, attempt = W.bpe(data, off, span=span)
    assert st == 0
    exp = [r['ids_' + name] for r in rows]
    exp_splits = np.zeros(len(rows) + 1, dtype=np.int64)
    np.cumsum([len(e) for e in exp], out=exp_splits[1:])
    assert np.array_equal(splits, exp_splits)
    assert ids.tolist() == [i for e in exp for i in e]


def test_bpe_small_stage_and_random_spans(golden, bpe_rows, models_dir):
    W.load_bpe(os.path.join(models_dir, 'bpe24k.json'))
    rows = _walker_rows(bpe_rows)
    lines = [r['norm'] for r in rows] + ['', '', '']
    exp = [r['ids_bpe24k'] for r in rows] + [[2, 3]] * 3
    data, off = sc.pack(lines)
    ids, splits, st, _ = W.bpe(data, off, span=50, rng=np.random.default_rng(1), stage_cap=3)
    assert st == 0
    assert ids.tolist() == [i for e in exp for i in e]
    assert splits[-1] == len(ids)


def test_bpe_renormalizes_when_needed(models_dir):
    # text that is NOT in NFC (what normalize_text can leave behind after filtering: U+0928 + U+093C adjacent)
    m = O.BpeModel(os.path.join(models_dir, 'bpe24k.json'))
    W.load_bpe(os.path.join(models_dir, 'bpe24k.json'))
    lines = ['ऩ क्ष', 'abc', 'ऱा', 'x']
    data, off = sc.pack(lines)
    ids, splits, st, attempt = W.bpe(data, off, span=16)
    assert attempt == 1 and st == 0
    exp = [O.bpe_encode(m, s) for s in lines]
    assert ids.tolist() == [i for e in exp for i in e]


def test_bpe_long_word_uses_pool(models_dir):
    m = O.BpeModel(os.path.join(models_dir, 'bpe24k.json'))
    W.load_bpe(os.path.join(models_dir, 'bpe24k.json'))
    lines = ['ab' * 200 + ' ' + 'कख' * 90, 'ok']
    data, off = sc.pack(lines)
    ids, splits, st, _ = W.bpe(data, off, span=32)
    assert st == 0
    exp = [O.bpe_encode(m, s) for s in lines]
    assert ids.tolist() == [i for e in exp for i in e]


@pytest.mark.parametrize('name', ['spm24k', 'spm_corpus'])
def test_unigram_ids_match_reference(golden, models_dir, name):
    assert W.load_spm(os.path.join(models_dir, name + '.model')) == golden['vocab_size'][name]
    rows = _rows(golden)
    data, off = sc.pack([r['norm'] for r in rows])
    ids, splits = W.unigram(data, off)
    exp = [r['ids_' + name] for r in rows]
    exp_splits = np.zeros(len(rows) + 1, dtype=np.int64)
    np.cumsum([len(e) for e in exp], out=exp_splits[1:])
    assert np.array_equal(splits, exp_splits)
    assert ids.tolist() == [i for e in exp for i in e]


def test_signature_matches_reference(golden):
    words = list(golden['signature'].keys())
    data, off = sc.pack(words)
    out, out_off = W.signature(data, off)
    b = out.tobytes()
    got = [b[out_off[i]:out_off[i + 1]].decode('utf-8') for i in range(len(words))]
    assert got == [golden['signature'][w] for w in words]


def test_loader_rejects_unsupported(models_dir, tmp_path):
    import json
    j = json.load(open(os.path.join(models_dir, 'bpe_corpus.json'), encoding='utf-8'))
    j['pre_tokenizer'] = {'type': 'ByteLevel'}
    p = str(tmp_path / 'bad.json')
    with open(p, 'w') as f:
        json.dump(j, f)
    with pytest.raises(ValueError):
        W.load_bpe(p)
    open(p, 'wb').write(b'\x00\x01garbage')
    with pytest.raises(ValueError):
        W.load_spm(p)


def _flat(exp):
    sp = np.zeros(len(exp) + 1, dtype=np.int64)
    np.cumsum([len(e) for e in exp], out=sp[1:])
    return [i for e in exp for i in e], sp


@pytest.mark.parametrize('real,cache_bits,prewarm', [(30, 14, 1), (1, 4, 0), (3, 8, 1), (30, 2, 0)])
def test_bpe_event_stream(golden, bpe_rows, models_dir, real, cache_bits, prewarm):
    """ak_tok.cuh, BPE: lanes -> word / row events -> word cache (tiny tables force probing and uncached words) -> ids
    == the reference's ids"""
    W.load_bpe(os.path.join(models_dir, 'bpe24k.json'))
    rows = bpe_rows
    lines = [r['norm'] for r in rows] + ['', '', 'ab' * 200 + ' ' + '\u0915\u0916' * 90, '', 'a_b9 \u0964\u0965\u0970\u0966 x', '\t \n']
    m = O.BpeModel(os.path.join(models_dir, 'bpe24k.json'))
    exp = [r['ids_bpe24k'] for r in rows] + [O.bpe_encode(m, s) for s in lines[len(rows):]]
    data, off = sc.pack(lines)
    ids, splits, st, stats = W.tok(0, data, off, real=real, cache_bits=cache_bits, prewarm=prewarm)
    assert st == 0
    flat, sp = _flat(exp)
    assert np.array_equal(splits, sp)
    assert ids.tolist() == flat
    # compact outputs: uint16 ids, int32 splits
    ids16, sp32, st, _ = W.tok(0, data, off, real=real, cache_bits=cache_bits, prewarm=prewarm, u16=True, splits_i32=True)
    assert st == 0 and ids16.dtype == np.uint16 and ids16.tolist() == flat and np.array_equal(sp32, sp)
    # too few event slots per warp tile: refused with the number that was needed, and that number works
    _, _, st, stats = W.tok(0, data, off, real=30, cap=40)
    assert st & 1 and stats['slots_needed'] > 40
    ids, splits, st, _ = W.tok(0, data, off, real=30, cap=(stats['slots_needed'] + 3) & ~3)
    assert st == 0 and ids.tolist() == flat


def test_bpe_event_stream_long_words(models_dir):
    """words longer than the boundary masks a lane can see (its own 32 bytes + the next two lanes'): every alignment of
    the word end against the lanes, including the right halo lane whose last two bytes are not classified"""
    W.load_bpe(os.path.join(models_dir, 'bpe24k.json'))
    m = O.BpeModel(os.path.join(models_dir, 'bpe24k.json'))
    rng = np.random.default_rng(11)
    lines = []
    for _ in range(400):
        parts = []
        for _ in range(int(rng.integers(1, 6))):
            n = int(rng.integers(40, 120))
            parts.append(('ab' * 80)[:n] if rng.random() < 0.5 else ('\u0915\u0916' * 40)[:n // 3])
            parts.append('.' if rng.random() < 0.5 else ' ')
            parts.append('c' * int(rng.integers(0, 3)))
        lines.append(''.join(parts))
    # a word that starts in the warp's last-but-one real lane and ends exactly where the halo lane's mask stops
    for s0 in range(896, 928, 3):
        for end in (988, 989, 990, 991, 992):
            lines.append('y' * (s0 - 2) + '. ' + 'a' * (end - s0) + '.' + 'c' * 20)
    data, off = sc.pack(lines)
    exp = [O.bpe_encode(m, s) for s in lines]
    for real in (30, 5):
        ids, splits, st, _ = W.tok(0, data, off, real=real)
        assert st == 0
        assert ids.tolist() == [i for e in exp for i in e]
    # the crafted rows again, each as its own batch: the row then starts at byte 0 of the first warp
    for s in lines[-55:]:
        data, off = sc.pack([s])
        ids, splits, st, _ = W.tok(0, data, off, real=30)
        assert st == 0 and ids.tolist() == O.bpe_encode(m, s)


def test_bpe_bit_parallel_classes_match_the_tables():
    """the plane logic hard-codes HF's pre-tokenizer classes and the encoder's alphabet for ASCII and U+0900-097F"""
    T = O.tables()
    m = None
    for cp in list(range(0x80)) + list(range(0x900, 0x980)):
        s = 'a' + chr(cp) + 'a'
        data, off = sc.pack([s])
        # class of the middle code point from the boundaries the front end finds: compare through the encoder below
        assert T.bpe_safe[cp] == (cp != 0x3C), hex(cp)
    assert not T.bpe_safe[0x9FE]


def test_bpe_rows_that_are_not_nfc_are_fixed_row_by_row(models_dir):
    """a row NFC would change is normalized and encoded on its own (row fix); the others stay on the fast path"""
    m = O.BpeModel(os.path.join(models_dir, 'bpe24k.json'))
    W.load_bpe(os.path.join(models_dir, 'bpe24k.json'))
    lines = ['\u0928\u093c \u0915\u094d\u0937', 'abc', '\u0930\u093c\u093e', 'x', '', 'kya \u0928\u093c haal']
    data, off = sc.pack(lines)
    exp = [O.bpe_encode(m, s) for s in lines]
    ids, splits, st, stats = W.tok(0, data, off)
    assert st == 0 and stats['flagged_rows'] == 3
    flat, sp = _flat(exp)
    assert ids.tolist() == flat and np.array_equal(splits, sp)
    ids, splits, st, attempt = W.bpe(data, off)
    assert attempt == 1 and st == 0 and ids.tolist() == flat


@pytest.mark.parametrize('real,cache_bits,prewarm', [(30, 14, 1), (1, 4, 0), (7, 9, 1)])
def test_unigram_event_stream(golden, models_dir, real, cache_bits, prewarm):
    """ak_tok.cuh, Unigram: words -> cached word lattices (robustness test against the score accumulated before the
    word, exact row Viterbi otherwise) == SentencePiece's ids"""
    W.load_spm(os.path.join(models_dir, 'spm24k.model'))
    rows = golden['rows']
    lines = [r['norm'] for r in rows]
    data, off = sc.pack(lines)
    ids, splits, st, stats = W.tok(1, data, off, real=real, cache_bits=cache_bits, prewarm=prewarm)
    assert st == 0
    flat, sp = _flat([r['ids_spm24k'] for r in rows])
    assert np.array_equal(splits, sp)
    assert ids.tolist() == flat
    print(stats)


def test_unigram_event_stream_exotic_rows(golden_raw, models_dir):
    """literal U+2581, rows longer than the word-wise path takes, other white space, leading / trailing / repeated spaces"""
    W.load_spm(os.path.join(models_dir, 'spm24k.model'))
    um = O.UnigramModel(os.path.join(models_dir, 'spm24k.model'))
    rows = golden_raw['rows']
    lines = [r['norm_nc'] for r in rows]
    extra = ['a\u2581b', '\u2581', 'x \u2581', ' \u2581y', 'a\u2581', '  lead', 'trail  ', 'a   b', '\ta\tb ', ' ', '', '\u00a0x',
             ' '.join(['\u0915\u092e\u0932', 'kya', 'haal'] * 1500), 'z' * 70 + ' ' + '\u0915' * 80, 'a' * 9000]
    data, off = sc.pack(lines + extra)
    ids, splits, st, stats = W.tok(1, data, off)
    assert st == 0
    exp = [r['ids_spm24k'] for r in rows] + [O.unigram_encode(um, s) for s in extra]
    flat, sp = _flat(exp)
    assert np.array_equal(splits, sp)
    assert ids.tolist() == flat
    assert stats['flagged_rows'] >= 7


def test_unigram_near_ties_take_the_exact_viterbi(models_dir):
    """rows made long enough that the accumulated score makes cached word lattices untrustworthy: those words are
    solved again by the exact row Viterbi, and the ids still equal SentencePiece's"""
    W.load_spm(os.path.join(models_dir, 'spm24k.model'))
    um = O.UnigramModel(os.path.join(models_dir, 'spm24k.model'))
    base = sc.Corpus('hindi', 5).lines(60000)
    lines = [' '.join(base[i:i + 25]) for i in range(0, len(base) - 25, 25)]       # ~6 KB rows (below the long-row limit)
    lines = [s for s in lines if len(s.encode('utf-8')) <= 8000]
    data, off = sc.pack(lines)
    ids, splits, st, stats = W.tok(1, data, off)
    assert st == 0
    assert stats['exact_words'] > 0
    exp = [O.unigram_encode(um, s) for s in lines]
    flat, sp = _flat(exp)
    assert np.array_equal(splits, sp) and ids.tolist() == flat


def test_raw_mode_cores(golden_raw, models_dir):
    T = O.tables()
    W.load_bpe(os.path.join(models_dir, 'bpe24k.json'))
    W.load_spm(os.path.join(models_dir, 'spm24k.model'))
    rows = golden_raw['rows']
    data, off = sc.pack([r['norm_nc'] for r in rows])
    ids, splits = W.unigram(data, off)
    assert ids.tolist() == [i for r in rows for i in r['ids_spm24k']]
    safe = [r for r in rows if all(T.bpe_safe[ord(c)] for c in r['norm_nc'])]
    data, off = sc.pack([r['norm_nc'] for r in safe])
    ids, splits, st, _ = W.bpe(data, off)
    assert st == 0 and ids.tolist() == [i for r in safe for i in r['ids_bpe24k']]
    # the event-stream encoder takes every row: added tokens in the raw text, compatibility characters, marks HF's older
    # Unicode tables order differently -- those rows go through the exact row path (HF's NFKC + added-token split)
    for key_in, key_ids in ((lambda r: r['norm_nc'], 'ids_bpe24k'),
                            (lambda r: O.normalize_text(r['in'], normalize_roman=False, clean_hinglish=False), 'ids_bpe24k_raw')):
        lines = [key_in(r) for r in rows]
        data, off = sc.pack(lines)
        for real, capb in ((30, 14), (3, 6)):
            ids, splits, st, stats = W.tok(0, data, off, real=real, cache_bits=capb)
            assert st == 0
            exp = [r[key_ids] for r in rows]
            assert splits.tolist() == np.concatenate(([0], np.cumsum([len(e) for e in exp]))).tolist()
            assert ids.tolist() == [i for e in exp for i in e]
    assert stats['flagged_rows'] > 300 and stats['flagged_rows'] < len(rows) // 2
    # the span walker on its own still refuses them (status bit 8 = AKSHAR_ST_ALPHABET)
    data, off = sc.pack(['ok', 'x\ufb01y', '<s>'])
    assert W.bpe(data, off)[2] & 8
    ids, splits, st, _ = W.tok(0, data, off)
    m = O.BpeModel(os.path.join(models_dir, 'bpe24k.json'))
    assert st == 0 and ids.tolist() == [i for t in ('ok', 'x\ufb01y', '<s>') for i in O.bpe_encode(m, t)]


# ---- ids -> text (ak_decode.cuh; reference tokenizer.py:195-246) ------------------------------------------------------
@pytest.mark.parametrize('name,kind', [('spm24k', 1), ('spm_corpus', 1), ('bpe24k', 0), ('bpe_corpus', 0)])
def test_decode_cores_against_the_reference(decode_fuzz, golden, models_dir, name, kind):
    """the piece tables, the row marks and the byte-run rule on the CPU, against what the unmodified reference decoded"""
    (W.load_spm if kind == 1 else W.load_bpe)(os.path.join(models_dir, name + ('.model' if kind == 1 else '.json')))
    F = decode_fuzz[name]
    got, st = W.decode(kind, 0, F['ids'])
    assert st == 0
    assert [g.decode('utf-8') for g in got] == F['decode']
    got, st = W.decode(kind, 1, F['ids_detok'] if kind == 0 else F['ids'])
    assert st == 0
    assert [g.decode('utf-8') for g in got] == F['detokenize']
    if name in ('spm24k', 'bpe24k'):
        rows = golden['rows'][:1500]
        got, st = W.decode(kind, 0, [r['ids_' + name] for r in rows])
        assert st == 0 and [g.decode('utf-8') for g in got] == [r['dec_' + name] for r in rows]
        got, st = W.decode(kind, 1, [r['ids_' + name] for r in rows])
        assert st == 0 and [g.decode('utf-8') for g in got] == [r['detok_' + name] for r in rows]
    if kind == 1:
        _, st = W.decode(kind, 0, [[5, 10 ** 6]])
        assert st == 128                                               # AKSHAR_ST_BAD_ID: DecodeIds raises IndexError


# ---- model loaders refuse what they cannot represent (ak_models.cpp) ---------------------------------------------------
def test_malformed_models_are_refused(models_dir, tmp_path):
    """ids outside [0, 2^24), non-integral ids, template ids the vocabulary does not hold, added-token options the device
    matcher does not implement, truncated files: an error string, never a crash (the C ABI wraps the loaders in try/catch
    and returns AKSHAR_E_MODEL)"""
    import json
    good = json.load(open(os.path.join(models_dir, 'bpe_corpus.json'), encoding='utf-8'))

    def load(j):
        p = tmp_path / 'm.json'
        p.write_text(json.dumps(j, ensure_ascii=False), encoding='utf-8')
        return W.load_bpe(str(p))

    assert load(good) == len(set(good['model']['vocab'].values()) | {t['id'] for t in good['added_tokens']})
    for mutate in (lambda j: j['model']['vocab'].__setitem__('zz', -5),
                   lambda j: j['model']['vocab'].__setitem__('zz', 1 << 40),
                   lambda j: j['model']['vocab'].__setitem__('zz', 7.5),
                   lambda j: j['added_tokens'][0].__setitem__('id', -1),
                   lambda j: j['added_tokens'][0].__setitem__('single_word', True),
                   lambda j: j['added_tokens'][0].__setitem__('content', ''),
                   lambda j: j['post_processor']['special_tokens']['<s>'].__setitem__('ids', [1 << 30]),
                   lambda j: j['model'].__setitem__('merges', ['a']),
                   lambda j: j.__setitem__('model', {'type': 'WordPiece'})):
        j = json.loads(json.dumps(good))
        mutate(j)
        with pytest.raises(ValueError):
            load(j)
    raw = open(os.path.join(models_dir, 'bpe_corpus.json'), 'rb').read()
    (tmp_path / 't.json').write_bytes(raw[:len(raw) // 2])
    with pytest.raises(ValueError):
        W.load_bpe(str(tmp_path / 't.json'))
    spm = open(os.path.join(models_dir, 'spm_corpus.model'), 'rb').read()
    for cut in (0, 1, 7, len(spm) // 3, len(spm) - 3):
        (tmp_path / 't.model').write_bytes(spm[:cut])
        try:
            W.load_spm(str(tmp_path / 't.model'))          # a prefix that happens to parse is fine; a crash is not
        except ValueError:
            pass
    (tmp_path / 't.model').write_bytes(b'\xff' * 64)
    with pytest.raises(ValueError):
        W.load_spm(str(tmp_path / 't.model'))
    W.load_bpe(os.path.join(models_dir, 'bpe24k.json'))
    W.load_spm(os.path.join(models_dir, 'spm24k.model'))


def test_zalgo_rows_through_the_event_stream_encoders(models_dir):
    """rows with up to 240 stacked marks on a base (NFC-normalized, as the encoders get them from normalize_text): the
    event-stream cores (words, row fix, resolve, emit) give the oracle's ids for both models"""
    import random
    rng = random.Random(11)
    marks = [chr(c) for c in (0x300, 0x301, 0x302, 0x303, 0x308, 0x30a, 0x316, 0x317, 0x323, 0x324, 0x325, 0x327, 0x328, 0x32d,
                              0x334, 0x335, 0x336, 0x338, 0x345, 0x35c, 0x360, 0x489, 0x93c, 0x94d, 0x951, 0x952)]
    lines = []
    for i in range(120):
        parts = []
        for _ in range(rng.choice((1, 3, 8))):
            base = rng.choice('aeou AEH\u0915\u0930\u0928z')
            k = rng.choice((0, 1, 5, 20, 45, 70, 120, 200, 240))
            parts.append(base + ''.join(rng.choice(marks) for _ in range(k)))
        lines.append(' '.join(parts))
    raw = [O.normalize_text(t, True, False) for t in lines]       # marks kept
    clean = [O.normalize_text(t) for t in lines]                  # marks dropped by the allow-list
    mb = O.BpeModel(os.path.join(models_dir, 'bpe24k.json'))
    mu = O.UnigramModel(os.path.join(models_dir, 'spm24k.model'))
    for rows in (raw, clean):
        data, off = sc.pack(rows)
        W.load_bpe(os.path.join(models_dir, 'bpe24k.json'))
        ids, splits, st, _ = W.tok(0, data, off)
        flat, sp = _flat([O.bpe_encode(mb, s) for s in rows])
        assert st == 0 and np.array_equal(splits, sp) and ids.tolist() == flat
        W.load_spm(os.path.join(models_dir, 'spm24k.model'))
        ids, splits, st, _ = W.tok(1, data, off)
        flat, sp = _flat([O.unigram_encode(mu, s) for s in rows])
        assert st == 0 and np.array_equal(splits, sp) and ids.tolist() == flat


def wide_unicode_encoder_lines():
    """1500 rows drawn from 27 blocks (compatibility forms HF's NFKC rewrites, marks, Hangul, full-width forms, mathematical
    alphanumerics, enclosed characters ...) with added-token syntax sprinkled in, normalized with `clean_hinglish=False`"""
    import random
    import unicodedata as u
    rng = random.Random(77)
    blocks = [(0x20, 0x7f), (0x20, 0x7f), (0xa0, 0x17f), (0x300, 0x36f), (0x370, 0x3ff), (0x590, 0x5ff), (0x600, 0x6ff),
              (0x900, 0x97f), (0x900, 0x97f), (0x980, 0x9ff), (0xe00, 0xe7f), (0xf00, 0xfff), (0x1100, 0x11ff), (0x1e00, 0x1eff),
              (0x2000, 0x206f), (0x2100, 0x214f), (0x2460, 0x24ff), (0x3040, 0x30ff), (0x3300, 0x33ff), (0xac00, 0xd7ff),
              (0xf900, 0xfaff), (0xfb00, 0xfb4f), (0xfe00, 0xfe0f), (0xff00, 0xffef), (0x1d400, 0x1d7ff), (0x1f100, 0x1f1ff),
              (0x1f300, 0x1f6ff)]

    def rcp():
        while True:
            a, b = rng.choice(blocks)
            c = rng.randint(a, b)
            if 0xd800 <= c <= 0xdfff or (u.category(chr(c)) == 'Cn' and rng.random() < 0.9):
                continue
            return chr(c)
    lines = []
    for i in range(1500):
        n = rng.choice((1, 2, 5, 12, 30, 60))
        pool = [rcp() for _ in range(rng.choice((2, 4, 8)))] + [' ', '<s>', '</s>', '<unk>', '<']
        s = ''.join(rng.choice(pool) if rng.random() < 0.6 else rcp() for _ in range(n))
        lines.append(s.replace('\n', ' ').replace('\r', ' ').replace('\x00', ' '))
    return [O.normalize_text(s, True, False) for s in lines]


def test_wide_unicode_fuzz_through_the_encoders(models_dir, library_fuzz):
    """wide-Unicode rows: the oracle gives the ids the libraries the reference calls (tokenizers, sentencepiece) returned
    for them (recorded by tools/make_golden_fuzz.py), and the event-stream cores give the oracle's"""
    norm = wide_unicode_encoder_lines()
    ref = library_fuzz['encoders']
    assert norm == ref['rows'], 'the generated rows are not the recorded ones'
    mb = O.BpeModel(os.path.join(models_dir, 'bpe24k.json'))
    mu = O.UnigramModel(os.path.join(models_dir, 'spm24k.model'))
    exp_b = [O.bpe_encode(mb, s) for s in norm]
    exp_u = [O.unigram_encode(mu, s) for s in norm]
    assert exp_b == ref['bpe24k']
    assert exp_u == ref['spm24k']
    data, off = sc.pack(norm)
    W.load_bpe(os.path.join(models_dir, 'bpe24k.json'))
    ids, splits, st, _ = W.tok(0, data, off)
    flat, sp_ = _flat(exp_b)
    assert st == 0 and np.array_equal(splits, sp_) and ids.tolist() == flat
    W.load_spm(os.path.join(models_dir, 'spm24k.model'))
    ids, splits, st, _ = W.tok(1, data, off)
    flat, sp_ = _flat(exp_u)
    assert st == 0 and np.array_equal(splits, sp_) and ids.tolist() == flat
