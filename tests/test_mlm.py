"""Masked language-model batches (DataCollatorForLanguageModeling's 80/10/10 masking with Philox draws keyed by seed,
epoch, row and position): the oracle (tools/mlm_oracle.py) against what transformers' collator returned with those draws
(tests/golden/mlm_hf.json.gz, tools/make_golden_mlm.py), the AK_HD arithmetic of the kernel (ak_mlm.cuh, built on the CPU
with tests/csrc/mlm_shim.cpp) against the oracle, and the device path (Engine.mlm_mask, aksharTokenizer.encode_batch_mlm,
corpus.pack_lines(mlm=...)) against both."""
import ctypes
import gzip
import json
import math
import os
import random
import subprocess
import zlib

import numpy as np
import pytest

import mlm_oracle as O
import pack_oracle as P
import windows_oracle as W

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, 'tests', 'golden')
MODELS = os.path.join(GOLDEN, 'models')
KAT = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
       ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
       ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]


@pytest.fixture(scope='module')
def fix():
    with gzip.open(os.path.join(GOLDEN, 'mlm_hf.json.gz'), 'rb') as f:
        return json.loads(f.read().decode('utf-8'))


def crc(a):
    return zlib.crc32(np.ascontiguousarray(a, np.int64).tobytes())


def fixture_inputs(fix, golden):
    """name -> int64 [N, L] input_ids of every fixture input, rebuilt from the golden rows by the windows / pack oracles"""
    rows = [golden['rows'][i] for i in fix['rows']]
    out = {}
    for name, d in fix['inputs'].items():
        key = 'ids_%s' % d['model']
        if d['kind'] == 'windows':
            ids, _, _ = W.windows([r[key] for r in rows], 2, 3, d['max_length'], d['stride'], False, True, 'longest', None, False,
                                  d['pad_id'])
            ids = np.asarray(ids, np.int64)
        else:
            pieces, _ = P.pack([r[key] for r in rows], d['block_size'], d['eos_id'])
            ids = np.asarray(P.flatten(pieces)['input_ids'], np.int64).reshape(-1, d['block_size'])
        assert list(ids.shape) == d['shape'] and crc(ids) == d['crc'], name
        out[name] = ids
    return out


def calls(fix):
    """(input name, setting index, (p, m, r), key index, (seed, epoch, row_base), record) of every recorded call"""
    for name, recs in fix['calls'].items():
        for si, per_key in enumerate(recs):
            for ki, rec in enumerate(per_key):
                yield name, si, tuple(fix['settings'][si]), ki, tuple(fix['keys'][ki]), rec


def oracle_call(fix, name, ids, pmr, key):
    d = fix['inputs'][name]
    M = fix['models'][d['model']]
    seed, epoch, row_base = key
    return O.mask(ids, M['special'], M['V'], M['mask_id'], seed, *pmr, epoch=epoch, row_base=row_base, pad_id=d['pad_id'])


# ------------------------------------------------------------------ CPU: the oracle is the collator
def test_fixture_holds_every_configuration(fix):
    assert fix['pins'] == {'transformers': '5.5.0'}
    assert [tuple(s) for s in fix['settings']] == [(.15, .8, .1), (.3, .8, .1), (.15, 1, 0), (.5, 0, 1), (0, .8, .1), (1, .8, .1),
                                                   (.4, .5, .5), (.2, .7, 0)]
    assert [tuple(k) for k in fix['keys']] == [(0, 0, 0), (2 ** 64 - 1, 2 ** 32 - 1, 2 ** 32 - 3), (987654321, 7, 2 ** 40)]
    assert set(fix['inputs']) == {'windows_bpe24k', 'packed_bpe24k_256', 'packed_bpe24k_512', 'packed_spm24k_256', 'packed_spm24k_512'}
    assert fix['models'] == {'bpe24k': {'V': 24000, 'mask_id': 4, 'special': [0, 1, 2, 3, 4]},
                             'spm24k': {'V': 24000, 'mask_id': 3, 'special': [0, 1, 2, 3]}}
    assert all(len(recs) == 8 and all(len(k) == 3 for k in recs) for recs in fix['calls'].values())
    assert len(fix['verbatim']) == 2


def test_oracle_equals_collator(fix, golden):
    """every recorded call: the counts of selected / replaced / random positions and the CRC32 of input_ids and labels"""
    inputs = fixture_inputs(fix, golden)
    n = 0
    for name, si, pmr, ki, key, rec in calls(fix):
        out, labels, counts = oracle_call(fix, name, inputs[name], pmr, key)
        assert {'counts': list(counts), 'crc': {'input_ids': crc(out), 'labels': crc(labels)}} == rec, (name, pmr, key)
        n += 1
    assert n == 5 * 8 * 3


def test_oracle_equals_collator_verbatim(fix, golden):
    """the two calls stored verbatim (rows [a, b) of an input with row_base + a): the oracle's result, which is also rows
    a..b of the oracle's one call over the whole input"""
    inputs = fixture_inputs(fix, golden)
    for v in fix['verbatim']:
        a, b = v['rows']
        pmr, (seed, epoch, row_base) = tuple(fix['settings'][v['setting']]), tuple(fix['keys'][v['key']])
        out, labels, _ = oracle_call(fix, v['input'], inputs[v['input']][a:b], pmr, (seed, epoch, row_base + a))
        assert out.tolist() == v['input_ids'] and labels.tolist() == v['labels']
        whole, whole_labels, _ = oracle_call(fix, v['input'], inputs[v['input']], pmr, (seed, epoch, row_base))
        assert np.array_equal(whole[a:b], out) and np.array_equal(whole_labels[a:b], labels)


def test_philox_known_answers():
    for ctr, key, want in KAT:
        assert O.philox(ctr, key) == want
        got = O.philox_np(*[np.array([c], np.uint32) for c in ctr], *key)
        assert tuple(int(w[0]) for w in got) == want


def test_thresholds():
    """the one threshold function of the engine against the oracle's, at the ends, at 0.15 and where m + r = 1 in double
    makes r / (1 - m) fall either side of 1"""
    from akshar_b200.batch import mlm_thresholds
    assert mlm_thresholds(0, .8, .1)[0] == 0 and mlm_thresholds(1, .8, .1)[0] == 2 ** 32
    assert mlm_thresholds(.15, .8, .1) == (math.ceil(float(np.float32(.15)) * 2 ** 32), math.ceil(float(np.float32(.8)) * 2 ** 32),
                                           2 ** 31)
    assert mlm_thresholds(.15, .8, .1)[0] == 644245120 != math.ceil(.15 * 2 ** 32)
    assert .3 / (1 - .7) < 1 < .1 / (1 - .9)                  # m + r = 1: the ratio in double is not 1
    assert mlm_thresholds(.15, .7, .3)[2] == mlm_thresholds(.15, .9, .1)[2] == 2 ** 32
    assert mlm_thresholds(.15, 1, 0)[2] == mlm_thresholds(.15, .5, 0)[2] == 0 and mlm_thresholds(.15, 0, 1)[1:] == (0, 2 ** 32)
    for p, m, r in [(.15, .8, .1), (.3, .8, .1), (.15, 1, 0), (.5, 0, 1), (0, .8, .1), (1, .8, .1), (.4, .5, .5), (.2, .7, 0),
                    (.7, .3, .7), (1e-9, .1, .2), (.999999999, .25, .75)]:
        assert mlm_thresholds(p, m, r) == O.thresholds(p, m, r), (p, m, r)


# ------------------------------------------------------------------ CPU: the kernel's arithmetic is the oracle
@pytest.fixture(scope='module')
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp('mlm_shim') / 'libmlm_shim.so')
    subprocess.check_call(['g++', '-O2', '-std=c++17', '-shared', '-fPIC', '-o', so, os.path.join(ROOT, 'tests', 'csrc', 'mlm_shim.cpp')])
    lib = ctypes.CDLL(so)
    vp, i64, u64, u32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_uint64, ctypes.c_uint32
    lib.ms_philox.argtypes = [vp, vp, i64, vp]
    lib.ms_mask.argtypes = [vp, i64, i64, u64, u32, u64, vp, i64, i64, u32, vp, i64, vp]
    return lib


def shim_philox(shim, ctrs, keys):
    c = np.ascontiguousarray(ctrs, np.uint32)
    k = np.ascontiguousarray(keys, np.uint32)
    out = np.zeros_like(c)
    shim.ms_philox(c.ctypes.data, k.ctypes.data, c.shape[0], out.ctypes.data)
    return out


def test_shim_known_answers(shim):
    got = shim_philox(shim, [c for c, _, _ in KAT], [k for _, k, _ in KAT])
    assert [tuple(int(x) for x in r) for r in got] == [w for _, _, w in KAT]


def test_shim_equals_oracle_on_the_fixture(fix, golden, shim):
    inputs = fixture_inputs(fix, golden)
    for name, si, pmr, ki, key, rec in calls(fix):
        d = fix['inputs'][name]
        M = fix['models'][d['model']]
        ids = inputs[name].copy()
        labels = np.zeros_like(ids)
        special = np.zeros(M['V'], np.uint8)
        special[M['special']] = 1
        t = np.array(O.thresholds(*pmr), np.uint64)
        seed, epoch, row_base = key
        pad = -1 if d['pad_id'] is None else d['pad_id']
        shim.ms_mask(ids.ctypes.data, ids.shape[0], ids.shape[1], seed, epoch, row_base, t.ctypes.data, M['mask_id'], pad, M['V'],
                     special.ctypes.data, M['V'], labels.ctypes.data)
        assert {'input_ids': crc(ids), 'labels': crc(labels)} == rec['crc'], (name, pmr, key)


def test_shim_near_2_32_and_2_64_equals_oracle(shim):
    """seeded counters whose words sit at and around 2^32 - 1 (positions, the two halves of rows near 2^32 and 2^64, epochs)
    and keys near 2^64: the shim's blocks against the oracle's"""
    rng = random.Random(20261022)
    edge = lambda: rng.choice([0, 1, 2 ** 31, 2 ** 32 - 2, 2 ** 32 - 1, rng.randrange(2 ** 32)])      # noqa: E731
    ctrs, keys = [], []
    for _ in range(4000):
        R = rng.choice([2 ** 32 - 1 + rng.randint(-3, 3), 2 ** 64 - 1 - rng.randint(0, 5), rng.randrange(2 ** 64)])
        ctrs.append((edge(), R & 0xFFFFFFFF, R >> 32, edge()))
        seed = rng.choice([2 ** 64 - 1 - rng.randint(0, 5), 2 ** 32 - 1 + rng.randint(-2, 2), rng.randrange(2 ** 64)])
        keys.append((seed & 0xFFFFFFFF, seed >> 32))
    got = shim_philox(shim, ctrs, keys)
    for c, k, g in zip(ctrs, keys, got):
        assert tuple(int(x) for x in g) == O.philox(c, k), (c, k)
    np_got = O.philox_np(*[np.array([c[i] for c in ctrs], np.uint32) for i in range(4)], 0, 0)
    assert all(tuple(int(w[i]) for w in np_got) == O.philox(c, (0, 0)) for i, c in enumerate(ctrs[:200]))


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
def toks(A):
    return {'bpe24k': A.aksharTokenizer(os.path.join(MODELS, 'bpe24k.json'), 'bpe'),
            'spm24k': A.aksharTokenizer(os.path.join(MODELS, 'spm24k.model'), 'sentencepiece')}


def device_input(fix, golden, toks, name):
    """the fixture input built by the device path from the golden rows' texts"""
    d = fix['inputs'][name]
    tk = toks[d['model']]
    texts = [golden['rows'][i]['in'] for i in fix['rows']]
    if d['kind'] == 'windows':
        ids = tk.encode_batch_tensors(texts, truncation=True, max_length=d['max_length'], stride=d['stride'],
                                      return_overflowing_tokens=True)['input_ids']
    else:
        ids = tk.encode_batch_packed(texts, d['block_size'], eos_id=d['eos_id'])[0]['input_ids']
    assert list(ids.shape) == d['shape'] and crc(ids.cpu().numpy()) == d['crc'], name
    return ids


def mlm_kw(pmr, key):
    (p, m, r), (seed, epoch, row_base) = pmr, key
    return dict(seed=seed, mlm_probability=p, mask_replace_prob=m, random_replace_prob=r, epoch=epoch, row_base=row_base)


@pytest.mark.gpu
def test_mlm_mask_equals_fixture(A, fix, golden, toks):
    """Engine.mlm_mask over the windows / packed batches the device paths build from the golden rows, both models, every
    setting and key"""
    base = {name: device_input(fix, golden, toks, name) for name in fix['inputs']}
    for name, si, pmr, ki, key, rec in calls(fix):
        d = fix['inputs'][name]
        tk = toks[d['model']]
        x = base[name].clone()
        out, labels = tk._eng.mlm_mask(x, tk.model.kind, pad_id=d['pad_id'], **mlm_kw(pmr, key))
        assert out is x and labels.dtype == x.dtype and labels.shape == x.shape
        assert {'input_ids': crc(out.cpu().numpy()), 'labels': crc(labels.cpu().numpy())} == rec['crc'], (name, pmr, key)
        assert int((labels != -100).sum()) == rec['counts'][0]


@pytest.mark.gpu
def test_encode_batch_mlm_equals_fixture(A, fix, golden, toks):
    """encode_batch_mlm in both of run_mlm.py's modes: windows (the dict with labels added) and packed blocks ((batch,
    rest) with the masked-LM labels in place of the causal-LM ones)"""
    texts = [golden['rows'][i]['in'] for i in fix['rows']]
    for name, si, pmr, ki, key, rec in calls(fix):
        d = fix['inputs'][name]
        tk = toks[d['model']]
        if d['kind'] == 'windows':
            out = tk.encode_batch_mlm(texts, truncation=True, max_length=d['max_length'], stride=d['stride'],
                                      return_overflowing_tokens=True, **mlm_kw(pmr, key))
            assert list(out) == ['input_ids', 'attention_mask', 'overflow_to_sample_mapping', 'labels']
        else:
            out, rest = tk.encode_batch_mlm(texts, block_size=d['block_size'], eos_id=d['eos_id'], return_seq_idx=True,
                                            **mlm_kw(pmr, key))
            assert list(out) == ['input_ids', 'labels', 'position_ids', 'seq_idx']
            assert rest.values.numel() < d['block_size']
        assert {'input_ids': crc(out['input_ids'].cpu().numpy()), 'labels': crc(out['labels'].cpu().numpy())} == rec['crc'], (name, pmr)


def specials_of(toks, model):
    return {'bpe24k': [0, 1, 2, 3, 4], 'spm24k': [0, 1, 2, 3]}[model]


def check_np(out, labels, want):
    assert np.array_equal(out.cpu().numpy(), want[0]) and np.array_equal(labels.cpu().numpy(), want[1])


@pytest.mark.gpu
@pytest.mark.parametrize('kind,model', [('hinglish', 'bpe24k'), ('hindi', 'spm24k')])
def test_mlm_at_64mb_equals_numpy_oracle(A, toks, kind, model):
    """64 MB of synthetic text: Hinglish as windows 512 / stride 128 (BPE), Hindi as packed blocks of 2048 with eos 2
    (SentencePiece); the result equals the vectorised oracle position for position"""
    import torch
    import synth_corpus as sc
    tk = toks[model]
    eng = tk._eng
    data, off = sc.Corpus(kind, 64).generate(64 << 20)
    enc, _ = eng.tokenizer_encode_batch((torch.from_numpy(data), torch.from_numpy(off)), tk.model.kind)
    if model == 'bpe24k':
        ids = eng.windows_batch(enc, 0, max_length=512, truncation=True, stride=128, return_overflowing_tokens=True)['input_ids']
        pad = eng.pad_id(0)
    else:
        ids = eng.pack_batch(enc, 2048, eos_id=2)[0]['input_ids']
        pad = None
    assert ids.numel() > 4 << 20
    orig = ids.cpu().numpy()
    for pmr, key in (((.15, .8, .1), (12345, 3, 77)), ((.3, .5, .4), (2 ** 64 - 1, 2 ** 32 - 1, 2 ** 32 - 5))):
        x = ids.clone()
        out, labels = eng.mlm_mask(x, tk.model.kind, pad_id=pad, **mlm_kw(pmr, key))
        want = O.mask(orig, specials_of(toks, model), 24000, eng.mask_id(tk.model.kind), key[0], *pmr, epoch=key[1], row_base=key[2],
                      pad_id=pad)
        check_np(out, labels, want)


@pytest.mark.gpu
def test_mlm_statistics_on_the_1gib_batch(A, toks):
    """the 1 GiB Hinglish batch of bench.py as windows 512 / stride 128: no special or pad position is selected, labels
    hold the original id exactly where selected, unselected ids stay; the selected / replaced / random counts lie within
    6 sigma of their binomial expectations, the random ids pass a chi-square bound over the vocabulary, and two adjacent
    rows are both selected at one position at the rate p^2 within 6 sigma"""
    import torch
    import synth_corpus as sc
    tk = toks['bpe24k']
    eng = tk._eng
    data, off = sc.Corpus('hinglish', 20261018).generate(1 << 30)
    enc, _ = eng.tokenizer_encode_batch((torch.from_numpy(data), torch.from_numpy(off)), 0)
    del data, off
    ids = eng.windows_batch(enc, 0, max_length=512, truncation=True, stride=128, return_overflowing_tokens=True)['input_ids']
    del enc
    V, mask_id, pad = 24000, eng.mask_id(0), eng.pad_id(0)
    orig = ids.clone()
    out, labels = eng.mlm_mask(ids, 0, seed=20261022, pad_id=pad)
    special = orig <= 4                                          # <pad> <unk> <s> </s> <mask> are ids 0..4
    sel = labels != -100
    assert not bool((sel & special).any())
    assert torch.equal(labels[sel], orig[sel]) and torch.equal(out[~sel], orig[~sel])
    from akshar_b200.batch import mlm_thresholds
    q1, q2, q3 = (t / 2 ** 32 for t in mlm_thresholds(.15, .8, .1))
    n_elig, n_sel = int((~special).sum()), int(sel.sum())
    rep = sel & (out == mask_id)                                 # a random id equal to mask_id counts here: ~n_random / V of them
    rnd = sel & ~rep & (out != orig)                             # a random id equal to the original is missed: as many
    n_rep, n_rnd = int(rep.sum()), int(rnd.sum())

    def within(k, n, q):
        return abs(k - n * q) <= 6 * math.sqrt(n * q * (1 - q)) + 2 * n_sel / V
    assert within(n_sel, n_elig, q1) and within(n_rep, n_sel, q2) and within(n_rnd, n_sel - n_rep, q3), (n_elig, n_sel, n_rep, n_rnd)
    counts = torch.bincount(out[rnd], minlength=V).double().cpu().numpy()
    counts = np.delete(counts, mask_id)
    e = counts.sum() / counts.size
    chi2 = float(((counts - e) ** 2 / e).sum())
    dof = counts.size - 1
    assert abs(chi2 - dof) < 6 * math.sqrt(2 * dof), chi2
    both_elig = ~special[:-1] & ~special[1:]
    n_pairs, n_both = int(both_elig.sum()), int((sel[:-1] & sel[1:]).sum())
    assert abs(n_both - n_pairs * q1 * q1) <= 6 * math.sqrt(n_pairs * q1 * q1 * (1 - q1 * q1)), (n_both, n_pairs)
    assert ids.numel() > 150 << 20


@pytest.mark.gpu
def test_invariances(A, toks, tmp_path):
    """rows [a, b) with row_base = a are rows a..b of the one call; padding to a multiple of 8 changes nothing below the
    old width; the same arguments give the same result, another epoch different masks; pack_lines(mlm=...) over a file in
    pieces equals encode_batch_mlm(block_size=...) over its lines"""
    import torch
    import synth_corpus as sc
    from akshar_b200 import corpus
    tk = toks['bpe24k']
    eng = tk._eng
    texts = sc.Corpus('hinglish', 5).lines(4 << 20)
    kw = dict(truncation=True, max_length=61, stride=13, return_overflowing_tokens=True, padding='max_length')
    base = tk.encode_batch_tensors(texts, **kw)['input_ids']
    whole = tk.encode_batch_mlm(texts, 99, epoch=4, row_base=1000, **kw)
    n = base.shape[0]
    cuts = [0, 1, n // 3, n // 3 + 7, n - 1, n]
    for a, b in zip(cuts, cuts[1:]):
        x, lab = eng.mlm_mask(base[a:b].clone(), 0, 99, epoch=4, row_base=1000 + a, pad_id=0)
        assert torch.equal(x, whole['input_ids'][a:b]) and torch.equal(lab, whole['labels'][a:b]), (a, b)
    padded = tk.encode_batch_mlm(texts, 99, epoch=4, row_base=1000, pad_to_multiple_of=8, **kw)
    w = whole['input_ids'].shape[1]
    assert padded['input_ids'].shape[1] % 8 == 0 and padded['input_ids'].shape[1] > w
    assert torch.equal(padded['input_ids'][:, :w], whole['input_ids']) and torch.equal(padded['labels'][:, :w], whole['labels'])
    assert bool((padded['input_ids'][:, w:] == 0).all()) and bool((padded['labels'][:, w:] == -100).all())
    again = tk.encode_batch_mlm(texts, 99, epoch=4, row_base=1000, **kw)
    assert torch.equal(again['input_ids'], whole['input_ids']) and torch.equal(again['labels'], whole['labels'])
    other = tk.encode_batch_mlm(texts, 99, epoch=5, row_base=1000, **kw)
    assert not torch.equal(other['labels'], whole['labels'])
    # pack_lines in pieces against one call
    data, off = sc.Corpus('hinglish', 6).generate(24 << 20)
    path = tmp_path / 'corpus.txt'
    np.insert(data, off[1:-1], np.uint8(10)).tofile(str(path))
    mlm = dict(seed=7, mlm_probability=.3, epoch=2)
    got = list(corpus.pack_lines(tk, str(path), 512, chunk_bytes=4 << 20, mlm=mlm, return_seq_idx=True))
    assert len(got) >= 4
    one, _ = tk.encode_batch_mlm(corpus.read_rows(str(path)), block_size=512, **mlm)
    for k in ('input_ids', 'labels'):
        assert torch.equal(torch.cat([b[k] for b in got]), one[k]), k


@pytest.mark.gpu
def test_edges(A, toks):
    """N = 0, L = 0, an 8 MB row as one row and in blocks, odd sizes and an input not 16-byte aligned (the scalar path),
    p = 0 and p = 1"""
    import torch
    eng = toks['bpe24k']._eng
    dev = eng.device
    launches = eng.launch_count()
    for shape in ((0, 7), (5, 0), (0, 0)):
        x = torch.zeros(shape, dtype=torch.int64, device=dev)
        out, labels = eng.mlm_mask(x, 0, 1)
        assert out.shape == labels.shape == shape
    assert eng.launch_count() == launches
    rng = np.random.default_rng(9)
    row = rng.integers(0, 24000, 8 << 20)
    for shape, key in (((1, 8 << 20), (3, 1, 2 ** 64 - 1)), (((8 << 20) // 128, 128), (3, 1, 2 ** 32 - 100))):
        ids = row.reshape(shape)
        out, labels = eng.mlm_mask(torch.from_numpy(ids).to(dev), 0, key[0], epoch=key[1], row_base=key[2])
        check_np(out, labels, O.mask(ids, [0, 1, 2, 3, 4], 24000, 4, key[0], epoch=key[1], row_base=key[2]))
    # odd N L, and a view 8 bytes past a 16-byte boundary
    big = torch.from_numpy(rng.integers(-3, 24010, 7 * 3 + 3)).to(dev)
    for x in (big[:21].view(7, 3), big[1:22].view(7, 3), big[3:].view(7, 3)):
        want = O.mask(x.cpu().numpy(), [0, 1, 2, 3, 4], 24000, 4, 11, .5, .5, .5, pad_id=24005)
        check_np(*eng.mlm_mask(x, 0, 11, .5, .5, .5, pad_id=24005), want)
    ids = torch.from_numpy(rng.integers(0, 24000, (300, 77))).to(dev)
    out, labels = eng.mlm_mask(ids.clone(), 0, 5, mlm_probability=0)
    assert torch.equal(out, ids) and bool((labels == -100).all())
    out, labels = eng.mlm_mask(ids.clone(), 0, 5, mlm_probability=1)
    elig = ids > 4
    assert torch.equal(labels[elig], ids[elig]) and bool((labels[~elig] == -100).all())


@pytest.mark.gpu
def test_refusals_leave_the_engine_usable(A, toks, tmp_path):
    import torch
    from akshar_b200 import corpus
    tk = toks['bpe24k']
    eng = tk._eng
    dev = eng.device
    ids = torch.arange(5, 29, dtype=torch.int64, device=dev).view(4, 6)
    bad = [dict(mlm_probability=-.1), dict(mlm_probability=1.5), dict(mlm_probability=None),
           dict(mask_replace_prob=.9, random_replace_prob=.2), dict(mask_replace_prob=-.1), dict(random_replace_prob=-.1),
           dict(mask_replace_prob=-.5, random_replace_prob=1.2), dict(seed=-1), dict(seed=2 ** 64), dict(seed=1.0),
           dict(epoch=-1), dict(epoch=2 ** 32), dict(row_base=-1), dict(row_base=2 ** 64), dict(row_base=2 ** 64 - 3),
           dict(mask_id=24000), dict(mask_id=-1), dict(pad_id=-1), dict(pad_id=True)]
    for kw in bad:
        kw.setdefault('seed', 1)
        with pytest.raises(ValueError):
            eng.mlm_mask(ids.clone(), 0, **kw)
    for x in (ids.to(torch.int32), ids.view(-1), ids.t(), ids.cpu(), ids.tolist()):
        with pytest.raises(ValueError):
            eng.mlm_mask(x, 0, 1)
    # a model without <mask> and no mask_id
    j = json.load(open(os.path.join(MODELS, 'bpe24k.json'), encoding='utf-8'))
    j['added_tokens'] = [t for t in j['added_tokens'] if t['content'] != '<mask>']
    no_mask = A.Engine(dev.index)
    no_mask.load_bpe(json.dumps(j).encode('utf-8'))
    assert no_mask.mask_id(0) is None
    with pytest.raises(ValueError, match='mask token'):
        no_mask.mlm_mask(ids.clone(), 0, 1)
    assert no_mask.mlm_mask(ids.clone(), 0, 1, mlm_probability=1, mask_replace_prob=1, random_replace_prob=0, mask_id=7)[0].eq(7).all()
    with pytest.raises(A._lib.AksharCudaError):
        eng.mlm_mask(ids.clone(), 1, 1, mask_id=3)                # no SentencePiece model in this engine
    with pytest.raises(ValueError):
        tk.encode_batch_mlm(['a b'], 1, block_size=4, text_pair=['c'])
    path = tmp_path / 'two.txt'
    path.write_text('a b c\nd e f\n')
    with pytest.raises(ValueError):
        next(corpus.pack_lines(tk, str(path), 4, mlm=dict(seed=1, row_base=3)))
    x, labels = eng.mlm_mask(ids.clone(), 0, 1, mlm_probability=1)
    assert torch.equal(labels, ids)
