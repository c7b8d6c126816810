"""The encoders' word cache (akshar_b200/csrc/ak_wordcache.cuh) never changes an id.

CPU: a numpy restatement of the cache's hash against a g++ build of the header (tests/csrc/wordcache_shim.cpp), and an
exhausted probe chain on a host table.  GPU: the BPE and Unigram encoders against the reference vectors and the oracle
under every cache history -- just loaded, warm, restored past a quarter of the table, held and saturated, restored by
force while held, reloaded -- with akshar_word_cache_stats proving each state; words whose probe chain is full on a
nearly empty table; one new word inserted by hundreds of warps at once, read back in the next call."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import akshar_oracle as O
import synth_corpus as sc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODELS = os.path.join(ROOT, 'tests', 'golden', 'models')
BPE, SPM = os.path.join(MODELS, 'bpe24k.json'), os.path.join(MODELS, 'spm24k.model')
AKC_ENTRY, AKC_PROBES, AKC_BITS = 16, 16, 19
SLOTS = 1 << AKC_BITS

# ------------------------------------------------------------------ the hash, restated
_U = np.uint64


def _mix(h, k):
    h = (h ^ k) * _U(0xBF58476D1CE4E5B9)
    return (h << _U(27)) | (h >> _U(37))


def _fin(h):
    h = h ^ (h >> _U(31))
    h = h * _U(0xFF51AFD7ED558CCD)
    return h ^ (h >> _U(33))


def np_hash(words):
    """the hash akc_lookup4 computes for each word (bytes): its key words (8 bytes each, little endian, zero padded)
    mixed into 0x9E3779B97F4A7C15 + length, then finalised; a word's home slot is hash & (slots - 1)"""
    out = np.zeros(len(words), dtype=np.uint64)
    lens = np.array([len(w) for w in words], dtype=np.int64)
    for n in np.unique(lens):
        idx = np.flatnonzero(lens == n)
        nw = (int(n) + 7) // 8
        buf = np.zeros((idx.size, 8 * nw), dtype=np.uint8)
        buf[:, :n] = np.frombuffer(b''.join(words[i] for i in idx), dtype=np.uint8).reshape(idx.size, n)
        out[idx] = hash_keys(buf.view('<u8'), int(n))
    return out


def hash_keys(keys, n):
    """hashes of words of n bytes given as their key words ([N, ceil(n / 8)] uint64)"""
    with np.errstate(over='ignore'):
        h = np.full(keys.shape[0], _U(0x9E3779B97F4A7C15) + _U(n), dtype=np.uint64)
        for j in range(keys.shape[1]):
            h = _mix(h, keys[:, j].astype(np.uint64))
        return _fin(h)


def colliding_words(bits, count, n_candidates, seed, slot=None):
    """`count` or more distinct 8-letter lowercase words with the same home slot in a table of 2^bits entries (the
    fullest slot of n_candidates seeded words, or `slot`); no letter three times in a row, so normalize_text keeps them"""
    rng = np.random.default_rng(seed)
    keys = rng.integers(97, 123, size=(n_candidates, 8), dtype=np.uint8).view('<u8')[:, 0]
    home = (hash_keys(keys[:, None], 8) & _U((1 << bits) - 1)).astype(np.int64)
    if slot is None:
        slot = int(np.argmax(np.bincount(home, minlength=1 << bits)))
    words = sorted(set(k.tobytes() for k in keys[home == slot]))
    words = [w for w in words if not any(w[i] == w[i + 1] == w[i + 2] for i in range(6))]
    assert len(words) >= count
    return slot, words


# ------------------------------------------------------------------ CPU: the g++ build of the cache
@pytest.fixture(scope='module')
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp('wordcache_shim') / 'libwordcache_shim.so')
    subprocess.check_call(['g++', '-O1', '-std=c++17', '-shared', '-fPIC', '-o', so,
                           os.path.join(ROOT, 'tests', 'csrc', 'wordcache_shim.cpp')])
    lib = ctypes.CDLL(so)
    vp, u32, i32, i64 = ctypes.c_void_p, ctypes.c_uint32, ctypes.c_int, ctypes.c_int64
    lib.wc_lookup.argtypes = [vp, u32, ctypes.c_char_p, u32, vp]
    lib.wc_hash.argtypes = [ctypes.c_char_p, vp, i64, vp]
    lib.wc_insert.argtypes = [vp, u32, ctypes.c_char_p, u32, vp, i32, vp]
    lib.wc_insert.restype = i64
    lib.wc_get.argtypes = [vp, u32, ctypes.c_char_p, u32, vp]
    lib.wc_get.restype = i32
    return lib


def _ptr(a):
    return a.ctypes.data


def test_hash_restatement_equals_the_header(shim):
    """every key-word branch of akc_lookup4 (1, 2, 3, 4 words and the j >= 4 loop): words of 1 .. 56 bytes"""
    rng = np.random.default_rng(3)
    words = [rng.integers(0, 256, size=n, dtype=np.uint8).tobytes() for n in range(1, 57) for _ in range(24)]
    words += [b'a' * n for n in range(1, 57)] + [('क' * 18).encode()[:n] for n in range(1, 55)]
    off = np.zeros(len(words) + 1, dtype=np.int64)
    np.cumsum([len(w) for w in words], out=off[1:])
    got = np.zeros(len(words), dtype=np.uint64)
    shim.wc_hash(b''.join(words), _ptr(off), len(words), _ptr(got))
    assert np.array_equal(np_hash(words), got)
    # the home slot: where a word lands in an empty table
    bits = 12
    table = np.zeros((1 << bits) * AKC_ENTRY, dtype=np.uint64)
    r = np.zeros(3, dtype=np.int64)
    for w, h in zip(words[::7], got[::7]):
        shim.wc_lookup(_ptr(table), bits, w, len(w), _ptr(r))
        assert r[1] == -1 and r[2] == int(h) & ((1 << bits) - 1)


def test_exhausted_probe_chain_on_the_host_table(shim):
    """17 words with one home slot (near the end of the table: the chain wraps): the first 16 fill the chain, the 17th
    finds neither itself nor a free slot and inserting it changes nothing; the 16 still read back their ids"""
    bits = 10
    mask = (1 << bits) - 1
    home, words = colliding_words(bits, 17, 1 << 18, seed=5, slot=mask - 5)
    words = words[:17]
    table = np.zeros((1 << bits) * AKC_ENTRY, dtype=np.uint64)
    counter = np.zeros(1, dtype=np.uint64)
    ids = {w: np.arange(100 * i, 100 * i + (i % 15), dtype=np.int32) for i, w in enumerate(words)}   # 0 .. 14 ids
    slots = []
    for w in words[:16]:
        slots.append(shim.wc_insert(_ptr(table), bits, w, len(w), _ptr(ids[w]), ids[w].size, _ptr(counter)))
    assert slots == [(home + p) & mask for p in range(AKC_PROBES)]
    assert int(counter[0]) == 16
    r = np.zeros(3, dtype=np.int64)
    last = words[16]
    shim.wc_lookup(_ptr(table), bits, last, len(last), _ptr(r))
    assert r[1] == -1 and r[2] == -1 and int(r[0]) & mask == home
    before = table.copy()
    assert shim.wc_insert(_ptr(table), bits, last, len(last), _ptr(ids[last]), ids[last].size, _ptr(counter)) == -1
    assert np.array_equal(table, before) and int(counter[0]) == 16
    out = np.zeros(16, dtype=np.int32)
    for w in words[:16]:
        n = shim.wc_get(_ptr(table), bits, w, len(w), _ptr(out))
        assert n == ids[w].size and np.array_equal(out[:n], ids[w])
    assert shim.wc_get(_ptr(table), bits, last, len(last), _ptr(out)) == -1


# ------------------------------------------------------------------ GPU
@pytest.fixture(scope='module')
def A():
    import torch
    assert torch.cuda.is_available(), 'GPU tests need a CUDA device'
    import __graft_entry__ as g
    g.build()
    import akshar_b200
    return akshar_b200


@pytest.fixture(scope='module')
def oracles():
    return O.BpeModel(BPE), O.UnigramModel(SPM)


@pytest.fixture(scope='module')
def collide():
    """8-letter words that share one home slot of the 2^19-entry tables: at most 16 of them can ever be cached"""
    _, words = colliding_words(AKC_BITS, 24, 1 << 24, seed=19)
    return [w.decode() for w in words]


def new_engine(A, kind):
    """an engine of its own, so that no other test's cache history leaks in"""
    eng = A.Engine(0)
    (eng.load_bpe if kind == 0 else eng.load_spm)(BPE if kind == 0 else SPM)
    return eng


def stats(eng, kind):
    out = (ctypes.c_int64 * 4)()
    rc = eng.lib.akshar_word_cache_stats(eng._h, kind, ctypes.addressof(out), eng._stream())
    assert rc == 0, rc
    return [int(x) for x in out]


def roman_words(n, seed):
    """n distinct seeded lowercase words of 7 .. 12 letters without a letter three times in a row"""
    rng = np.random.default_rng(seed)
    m = n + n // 8 + 64
    a = rng.integers(0, 26, size=(m, 12), dtype=np.int64)
    for j in range(2, 12):
        t = (a[:, j] == a[:, j - 1]) & (a[:, j - 1] == a[:, j - 2])
        a[t, j] = (a[t, j] + 1) % 26
    a[np.arange(12)[None, :] >= rng.integers(7, 13, size=m)[:, None]] = -1
    _, first = np.unique(((a + 1) * 27 ** np.arange(12)).sum(1), return_index=True)
    a = a[np.sort(first)[:n]]
    keep = a >= 0
    blob = (a[keep] + 97).astype(np.uint8).tobytes().decode('ascii')
    off = np.concatenate([[0], np.cumsum(keep.sum(1))])
    return [blob[off[i]:off[i + 1]] for i in range(a.shape[0])]


_CONS = [chr(c) for c in range(0x0915, 0x0939) if c not in (0x0929, 0x0931, 0x0934)]
_MATRA = [''] + [chr(c) for c in (0x093E, 0x093F, 0x0940, 0x0941, 0x0942, 0x0947, 0x0948, 0x094B, 0x094C)]
_SYL = [c + m for c in _CONS for m in _MATRA]


def deva_words(n, seed):
    """n distinct seeded Devanagari words of 3 .. 5 syllables (consonant + optional vowel sign)"""
    rng = np.random.default_rng(seed)
    m = n + n // 8 + 64
    a = rng.integers(0, len(_SYL), size=(m, 5), dtype=np.int64)
    a[np.arange(5)[None, :] >= rng.integers(3, 6, size=m)[:, None]] = -1
    _, first = np.unique(((a + 1) * (len(_SYL) + 1) ** np.arange(5)).sum(1), return_index=True)
    return [''.join(_SYL[x] for x in row if x >= 0) for row in a[np.sort(first)[:n]]]


def host_batch(lines):
    import torch
    d, o = sc.pack(lines)
    return torch.from_numpy(d), torch.from_numpy(o)


def assert_rows(ids, exp_v, exp_sp, lines, what):
    v, sp = ids.values.cpu().numpy(), ids.splits.cpu().numpy()
    if np.array_equal(sp, exp_sp) and np.array_equal(v, exp_v):
        return
    for i in range(len(lines)):
        got, want = v[sp[i]:sp[i + 1]].tolist(), exp_v[exp_sp[i]:exp_sp[i + 1]].tolist()
        assert got == want, '%s: row %d %r' % (what, i, lines[i])
    assert False, what


def ragged(rows):
    sp = np.zeros(len(rows) + 1, dtype=np.int64)
    np.cumsum([len(r) for r in rows], out=sp[1:])
    return np.array([x for r in rows for x in r], dtype=np.int32), sp


@pytest.mark.gpu
@pytest.mark.parametrize('kind', [0, 1], ids=['bpe', 'unigram'])
def test_ids_do_not_depend_on_cache_history(A, golden, oracles, collide, kind):
    """the target batch (golden rows, words whose probe chain is full, seeded novel words) gives the reference / oracle
    ids in every state of the cache, and every row of every filler call equals a second engine's ids for the same rows
    (its cache restored before each call) and, on a seeded sample, the oracle's"""
    om, um = oracles
    words = roman_words if kind == 0 else deva_words
    model_ids = (lambda s: O.bpe_encode(om, s)) if kind == 0 else (lambda s: O.unigram_encode(um, s))
    key = 'ids_bpe24k' if kind == 0 else 'ids_spm24k'
    novel = words(12000, seed=100 + kind)
    extra = collide + [' '.join(collide)] + [' '.join(novel[i:i + 3]) for i in range(0, len(novel), 3)]
    target = [r['in'] for r in golden['rows']] + extra
    exp_v, exp_sp = ragged([r[key] for r in golden['rows']] + [model_ids(O.normalize_text(s)) for s in extra])
    h_target = host_batch(target)
    eng, twin = new_engine(A, kind), new_engine(A, kind)
    enc = eng.encode_bpe_batch if kind == 0 else eng.encode_unigram_batch
    enc2 = twin.encode_bpe_batch if kind == 0 else twin.encode_unigram_batch
    log = []

    def check_target(state):
        ids, _ = eng.tokenizer_encode_batch(h_target, kind)
        assert_rows(ids, exp_v, exp_sp, target, state)
        s = stats(eng, kind)
        log.append((state, s))
        return s

    seeds = iter(range(1000 + 100 * kind, 1100 + 100 * kind))

    def filler(n):
        seed = next(seeds)
        lines = words(n, seed)
        hb = host_batch(lines)
        got = enc(hb)
        twin.lib.akshar_word_cache_hold(twin._h, -1)
        ref = enc2(hb)
        import torch
        assert torch.equal(got.splits, ref.splits) and torch.equal(got.values, ref.values), 'filler %d' % seed
        pick = np.sort(np.random.default_rng(seed).choice(n, size=min(n, 20000), replace=False))
        v, sp = got.values.cpu().numpy(), got.splits.cpu().numpy()
        for i in pick:
            assert v[sp[i]:sp[i + 1]].tolist() == model_ids(lines[i]), 'filler %d row %d %r' % (seed, i, lines[i])
        s = stats(eng, kind)
        log.append(('filler of %d words' % n, s))
        return s

    def hold(h):
        assert eng.lib.akshar_word_cache_hold(eng._h, h) == 0

    try:
        # 1. just loaded (twice in a row: the words with a full probe chain miss on both calls)
        s0 = stats(eng, kind)
        log.append(('loaded', s0))
        assert s0[0] == SLOTS and 0 < s0[1] < SLOTS // 8 and s0[2] == 0 and s0[3] == 0
        learned = check_target('just loaded')[2]
        assert 0 < learned < SLOTS // 8
        fresh = learned + learned // 4          # what one target call learns on the image alone (races aside)
        # 2. warm: most words hit the entries the first call learned
        s = check_target('warm')
        assert learned <= s[2] <= learned + learned // 4
        # 3. past the quarter: the next call restores the image first
        s = filler(160000)
        assert s[2] > SLOTS // 4
        s = check_target('past the quarter')
        assert s[2] <= fresh
        # 4. held and saturated: long probe chains, most misses find no free slot
        hold(1)
        for _ in range(8):
            s = stats(eng, kind)
            if s[1] + s[2] >= 0.9 * SLOTS:
                break
            filler(250000)
        held = stats(eng, kind)
        assert held[1] + held[2] >= 0.9 * SLOTS and held[3] == 1
        s = check_target('held and saturated')
        assert s[2] >= held[2] and s[3] == 1
        hold(0)
        s = check_target('hold released')
        assert s[2] <= fresh and s[3] == 0
        # 5. a forced restore while held: the hold stays
        hold(1)
        s = filler(50000)
        assert s[2] > fresh
        hold(-1)
        s = check_target('forced restore while held')
        assert s[2] <= fresh and s[3] == 1
        s = check_target('held after the forced restore')
        assert s[2] >= log[-2][1][2] and s[3] == 1
        # 6. reload: a fresh image, no hold; the hold is the context's, so loading the other model clears it too
        (eng.load_bpe if kind == 0 else eng.load_spm)(BPE if kind == 0 else SPM)
        s = stats(eng, kind)
        assert s[1] == s0[1] and s[2] == 0 and s[3] == 0
        check_target('reloaded')
        hold(1)
        assert stats(eng, kind)[3] == 1
        (eng.load_spm if kind == 0 else eng.load_bpe)(SPM if kind == 0 else BPE)
        assert stats(eng, kind)[3] == 0 and stats(eng, 1 - kind)[3] == 0
        check_target('other model loaded')
    finally:
        for state, s in log:
            print('word cache %s %-32s slots %d image %d learned %d occupied %.3f hold %d' %
                  ('bpe' if kind == 0 else 'unigram', state, s[0], s[1], s[2], (s[1] + s[2]) / s[0], s[3]))


@pytest.mark.gpu
@pytest.mark.parametrize('kind', [0, 1], ids=['bpe', 'unigram'])
def test_exhausted_probe_chains(A, oracles, collide, kind):
    """words with one home slot on a nearly empty table: at most 16 are ever cached, the others miss with no free slot
    on their probe path in every call"""
    om, um = oracles
    model_ids = (lambda s: O.bpe_encode(om, s)) if kind == 0 else (lambda s: O.unigram_encode(um, s))
    eng = new_engine(A, kind)
    enc = eng.encode_bpe_batch if kind == 0 else eng.encode_unigram_batch
    lines = collide + [' '.join(collide), ' '.join(reversed(collide))]
    exp_v, exp_sp = ragged([model_ids(s) for s in lines])
    for call in range(2):
        assert_rows(enc(lines), exp_v, exp_sp, lines, 'call %d' % call)
        s = stats(eng, kind)
        assert 1 <= s[2] <= AKC_PROBES < len(collide)


@pytest.mark.gpu
@pytest.mark.parametrize('kind', [0, 1], ids=['bpe', 'unigram'])
def test_contended_insert(A, oracles, kind):
    """one new word of more than two ids in 100 k rows (between other new words): hundreds of warps race to publish it
    in one call; the next call reads the published entry (its ids 2.. from the entry's later sectors)"""
    om, um = oracles
    model_ids = (lambda s: O.bpe_encode(om, s)) if kind == 0 else (lambda s: O.unigram_encode(um, s))
    words = roman_words if kind == 0 else deva_words
    core = (lambda ids: ids[1:-1]) if kind == 0 else (lambda ids: ids)
    hot = next(w for w in words(200, seed=40 + kind) if 3 <= len(core(model_ids(w))) <= 14)
    others = words(26000, seed=50 + kind)
    others = [w for w in others if w != hot][:25000]
    lines = [hot if i % 4 else others[i // 4] + ' ' + hot for i in range(100000)]
    hot_ids = model_ids(hot)
    exp_v, exp_sp = ragged([hot_ids if i % 4 else model_ids(s) for i, s in enumerate(lines)])
    eng = new_engine(A, kind)
    enc = eng.encode_bpe_batch if kind == 0 else eng.encode_unigram_batch
    hb = host_batch(lines)
    assert_rows(enc(hb), exp_v, exp_sp, lines, 'racing call')
    learned = stats(eng, kind)[2]
    assert learned >= 1
    assert_rows(enc(hb), exp_v, exp_sp, lines, 'call after the race')
    assert_rows(enc([hot] * 3), *ragged([model_ids(hot)] * 3), [hot] * 3, 'the word alone')
