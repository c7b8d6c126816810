"""Model-ready sentence-pair windows (pair template, longest_first / only_first / only_second truncation with stride,
padding): the oracle (tools/windows_oracle.py, pair_windows) against what HF tokenizers returned
(tests/golden/pairs_hf.json.gz, tools/make_golden_pairs.py), the AK_HD pair plan of the kernels (ak_win.cuh, built on
the CPU with tests/csrc/pair_shim.cpp) against the oracle, and the device path (Engine.windows_batch(pair_ids=...),
aksharTokenizer.encode_batch_tensors(texts, text_pair=...)) against both."""
import ctypes
import gzip
import json
import os
import subprocess

import numpy as np
import pytest

from windows_oracle import pair_spans, pair_windows

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, 'tests', 'golden')
MODELS = os.path.join(GOLDEN, 'models')
VARIANTS = ('bpe24k', 'bpe24k_roberta', 'bpe24k_no_template')
STRATEGY_CODE = {'longest_first': 1, 'only_first': 2, 'only_second': 3}
# the oracle's refusals -> the kind of HF misbehaviour the fixture records
KIND_OF = (('too short', 'too_short'), ('stride', 'panic'), ('0 ids', 'wider'))


@pytest.fixture(scope='module')
def fix():
    with gzip.open(os.path.join(GOLDEN, 'pairs_hf.json.gz'), 'rb') as f:
        return json.loads(f.read().decode('utf-8'))


@pytest.fixture(scope='module')
def content(golden):
    return [r['ids_bpe24k'][1:-1] for r in golden['rows']]


def parse_trunc(name, P):
    """fixture name -> (max_length or None, stride, left)"""
    if name == 'none':
        return None, 0, False
    ml, st, d = name.split(',')
    return (P + int(ml[2:]) if ml.startswith('P+') else int(ml)), int(st), d == 'left'


def parse_pad(name):
    mode, side, mult = name.split(',')
    return mode, side == 'left', int(mult) or None


def batches(fix):
    n, b = len(fix['pairs']), fix['batch']
    return [(i, min(i + b, n)) for i in range(0, n, b)]


def n_template(V):
    return len(V['pre']) + len(V['mid']) + len(V['post'])


def oracle_kind(ca, cb, m, stride, strategy, left):
    """the oracle's windows of a pair as the fixture stores them: flat (startA, lenA, startB, lenB), or a refusal kind"""
    try:
        spans = pair_spans(ca, cb, m, stride, strategy, left, True)
    except ValueError as e:
        return next(k for key, k in KIND_OF if key in str(e))
    return [x for (a0, a1), (b0, b1) in spans for x in (a0, a1 - a0, b0, b1 - b0)]


def fixture_windows(V, fix, content, strategy, name, b0, b1, overflow=True):
    """HF's windows of the pairs b0..b1-1 (template ids included) and their pair numbers, from the recorded spans"""
    out, rows = [], []
    for p in range(b0, b1):
        a, b = fix['pairs'][p]
        sp = V['windows'][strategy][name][p]
        for k in range(0, len(sp) if overflow else 4, 4):
            out.append(V['pre'] + content[a][sp[k]:sp[k] + sp[k + 1]] + V['mid'] + content[b][sp[k + 2]:sp[k + 2] + sp[k + 3]] +
                       V['post'])
            rows.append(p - b0)
    return out, rows


def batch_refused(V, strategy, name, b0, b1):
    return any(isinstance(x, str) for x in V['windows'][strategy][name][b0:b1])


# ------------------------------------------------------------------ CPU: the oracle is HF
def test_fixture_holds_every_configuration(fix):
    assert fix['pins'] == {'tokenizers': '0.22.2', 'transformers': '5.5.0'}
    assert set(fix['variants']) == set(VARIANTS)
    assert fix['strategies'] == list(STRATEGY_CODE)
    assert len(fix['pairs']) == 640 and len(fix['trunc']) == 16 and len(fix['pad']) == 8 and len(fix['pad_trunc']) == 4
    for V in fix['variants'].values():
        for s in fix['strategies']:
            assert list(V['windows'][s]) == fix['trunc'] and list(V['batch_error'][s]) == fix['trunc']
            assert all(len(x) == 640 for x in V['windows'][s].values())
            assert all(len(x) == 10 for x in V['batch_error'][s].values())
            assert list(V['width'][s]) == fix['pad_trunc']
    kinds = {x for V in fix['variants'].values() for s in V['windows'].values() for w in s.values() for x in w if isinstance(x, str)}
    assert kinds == {'too_short', 'panic', 'wider'}
    assert len(fix['variants']['bpe24k']['verbatim']) == 2


@pytest.mark.parametrize('variant', VARIANTS)
def test_oracle_pairs_equal_hf(fix, content, variant):
    """every pair, strategy and configuration, refusals included; a batch HF refuses fails as its first refused pair"""
    V = fix['variants'][variant]
    P = n_template(V)
    for strategy in fix['strategies']:
        for name in fix['trunc']:
            ml, stride, left = parse_trunc(name, P)
            got = V['windows'][strategy][name]
            for p, (a, b) in enumerate(fix['pairs']):
                want = oracle_kind(len(content[a]), len(content[b]), None if ml is None else ml - P, stride, strategy, left)
                assert want == got[p], (variant, strategy, name, p)
            for bi, (b0, b1) in enumerate(batches(fix)):
                err = V['batch_error'][strategy][name][bi]
                kinds = [x for x in got[b0:b1] if isinstance(x, str)]
                assert err == (kinds[0] if kinds else None), (variant, strategy, name, bi)


@pytest.mark.parametrize('variant', VARIANTS)
def test_oracle_width_equals_hf(fix, content, variant):
    V = fix['variants'][variant]
    P = n_template(V)
    bos, eos = (2, 3) if V['template'] else (None, None)
    frame = (lambda c: [2] + c + [3]) if V['template'] else (lambda c: c)
    for strategy in fix['strategies']:
        for name in fix['pad_trunc']:
            ml, stride, left = parse_trunc(name, P)
            for pname, widths in V['width'][strategy][name].items():
                mode, pad_left, mult = parse_pad(pname)
                for bi, (b0, b1) in enumerate(batches(fix)):
                    ra = [frame(content[a]) for a, _ in fix['pairs'][b0:b1]]
                    rb = [frame(content[b]) for _, b in fix['pairs'][b0:b1]]
                    if widths[bi] is None:
                        with pytest.raises(ValueError):
                            pair_windows(ra, rb, bos, eos, V['pre'], V['mid'], V['post'], ml, stride, strategy, left, True, mode,
                                         mult, pad_left, 0, truncate=ml is not None)
                        continue
                    ids, _, _ = pair_windows(ra, rb, bos, eos, V['pre'], V['mid'], V['post'], ml, stride, strategy, left, True,
                                             mode, mult, pad_left, 0, truncate=ml is not None)
                    assert all(len(x) == widths[bi] for x in ids), (variant, strategy, name, pname, bi)


def test_oracle_equals_hf_verbatim(fix, content):
    V = fix['variants']['bpe24k']
    for rec in V['verbatim']:
        ml, stride, left = parse_trunc(rec['trunc'], 4)
        b0, b1 = batches(fix)[rec['batch']]
        ra = [[2] + content[a] + [3] for a, _ in fix['pairs'][b0:b1]]
        rb = [[2] + content[b] + [3] for _, b in fix['pairs'][b0:b1]]
        ids, mask, sample = pair_windows(ra, rb, 2, 3, [2], [3, 2], [3], ml, stride, rec['strategy'], left, True, rec['padding'],
                                         None, False, 0)
        assert ids == rec['input_ids'] and mask == rec['attention_mask'] and sample == rec['overflow_to_sample_mapping']


def test_oracle_refuses_what_hf_gets_wrong():
    with pytest.raises(ValueError):                     # no room left for content
        pair_windows([[2, 5, 3]], [[2, 6, 3]], 2, 3, [2], [3, 2], [3], 4, 0, 'longest_first', False, True, 'longest', None, False, 0)
    with pytest.raises(ValueError):                     # both sides must pair up
        pair_windows([[2, 5, 3]], [], 2, 3, [2], [3, 2], [3], 8, 0, 'longest_first', False, True, 'longest', None, False, 0)
    assert pair_spans(10, 3, 7, 1, 'only_first', False, True) == [((0, 4), (0, 3)), ((3, 7), (0, 3)), ((6, 10), (0, 3))]
    assert pair_spans(5, 5, 4, 0, 'longest_first', False, True)[:3] == [((0, 2), (0, 2)), ((2, 4), (0, 2)), ((2, 4), (2, 4))]
    assert len(pair_spans(5, 5, 4, 0, 'longest_first', False, True)) == 9
    assert pair_spans(2, 5, 4, 0, 'longest_first', False, False) == [((0, 2), (0, 2))]


# ------------------------------------------------------------------ CPU: the kernels' pair plan is the oracle
@pytest.fixture(scope='module')
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp('pair_shim') / 'libpair_shim.so')
    subprocess.check_call(['g++', '-O1', '-std=c++17', '-shared', '-fPIC', '-o', so, os.path.join(ROOT, 'tests', 'csrc', 'pair_shim.cpp'),
                           os.path.join(ROOT, 'akshar_b200', 'csrc', 'ak_models.cpp')])
    lib = ctypes.CDLL(so)
    lib.ps_pair_windows.restype = ctypes.c_int64
    lib.ps_pair_windows.argtypes = [ctypes.c_int64] * 4 + [ctypes.c_int] * 3 + [ctypes.c_void_p, ctypes.c_int64]
    lib.ps_load_pair.argtypes = [ctypes.c_char_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p]
    return lib


_PLAN_OUT = np.zeros(4 << 18, dtype=np.int64)


def plan_windows(shim, ca, cb, m, stride, strategy, left, overflow=True):
    out, cap = _PLAN_OUT, _PLAN_OUT.size // 4
    n = shim.ps_pair_windows(ca, cb, m, stride, STRATEGY_CODE[strategy], int(left), int(overflow), out.ctypes.data, cap)
    if n < 0:
        return {1: 'wider', 2: 'panic', 3: 'too_short'}[-n]
    assert n <= cap
    return [x for a0, a1, b0, b1 in out[:4 * n].reshape(-1, 4).tolist() for x in (a0, a1 - a0, b0, b1 - b0)]


@pytest.mark.parametrize('variant', VARIANTS)
def test_plan_equals_oracle_and_hf(fix, content, shim, variant):
    V = fix['variants'][variant]
    P = n_template(V)
    for strategy in fix['strategies']:
        for name in fix['trunc'][1:]:
            ml, stride, left = parse_trunc(name, P)
            for p, (a, b) in enumerate(fix['pairs']):
                got = plan_windows(shim, len(content[a]), len(content[b]), ml - P, stride, strategy, left)
                assert got == V['windows'][strategy][name][p], (variant, strategy, name, p)
                first = plan_windows(shim, len(content[a]), len(content[b]), ml - P, stride, strategy, left, overflow=False)
                assert first == (got if isinstance(got, str) else got[:4])
    # refusals the fixture cannot hold: more than 2^31 - 1 windows
    out = np.zeros(4, dtype=np.int64)
    assert shim.ps_pair_windows(70000, 70000, 2, 0, 1, 0, 1, out.ctypes.data, 1) == -4


def test_loader_parses_pair_slots(shim, tmp_path):
    base = json.load(open(os.path.join(MODELS, 'bpe24k.json'), encoding='utf-8'))
    s, e = {'SpecialToken': {'id': '<s>', 'type_id': 0}}, {'SpecialToken': {'id': '</s>', 'type_id': 1}}
    A, B = {'Sequence': {'id': 'A', 'type_id': 0}}, {'Sequence': {'id': 'B', 'type_id': 1}}

    def load(pair=None, drop=False, post=True):
        j = json.loads(json.dumps(base))
        if not post:
            j['post_processor'] = None
        elif drop:
            del j['post_processor']['pair']
        elif pair is not None:
            j['post_processor']['pair'] = pair
        raw = json.dumps(j).encode('utf-8')
        n = np.zeros(3, dtype=np.int32)
        ids = np.zeros(12, dtype=np.int32)
        ok = shim.ps_load_pair(raw, len(raw), n.ctypes.data, ids.ctypes.data)
        return ok, [ids[4 * k:4 * k + n[k]].tolist() for k in range(3)]

    assert load() == (1, [[2], [3, 2], [3]])                                  # the model's own template
    assert load([s, A, e, e, B, e]) == (1, [[2], [3, 3], [3]])                 # RoBERTa-style
    assert load(post=False) == (1, [[], [], []])                               # no post-processor
    assert load([A, B]) == (1, [[], [], []])
    assert load([s, s, s, s, A, B]) == (1, [[2, 2, 2, 2], [], []])
    for bad in ([s, s, s, s, s, A, B], [B, A], [A], [A, B, A], [s, A, {'SpecialToken': {'id': '<nope>', 'type_id': 0}}, B]):
        assert load(bad) == (0, [[], [], []]), bad                             # loads; only pair calls are refused
    assert load(drop=True) == (0, [[], [], []])


# ------------------------------------------------------------------ GPU
@pytest.fixture(scope='module')
def A():
    import torch
    assert torch.cuda.is_available(), 'GPU tests need a CUDA device'
    import __graft_entry__ as g
    g.build()
    import akshar_b200
    return akshar_b200


def variant_json(variant):
    j = json.load(open(os.path.join(MODELS, 'bpe24k.json'), encoding='utf-8'))
    if variant == 'bpe24k_no_template':
        j['post_processor'] = None
    elif variant == 'bpe24k_roberta':
        s, e = {'SpecialToken': {'id': '<s>', 'type_id': 0}}, {'SpecialToken': {'id': '</s>', 'type_id': 0}}
        j['post_processor']['pair'] = [s, {'Sequence': {'id': 'A', 'type_id': 0}}, e, e, {'Sequence': {'id': 'B', 'type_id': 0}}, e]
    return j


@pytest.fixture(scope='module')
def toks(A, tmp_path_factory):
    """one tokenizer per fixture variant"""
    d = tmp_path_factory.mktemp('pair_models')
    out = {}
    for v in VARIANTS:
        p = d / (v + '.json')
        p.write_text(json.dumps(variant_json(v)), encoding='utf-8')
        out[v] = A.aksharTokenizer(str(p), 'bpe')
    return out


def check_dense(out, want, want_rows, width, pad_left, pad_id, device, overflow=True):
    """the device tensors hold exactly the windows `want` (lists of ids), padded to `width`"""
    import torch
    ids, mask = out['input_ids'], out['attention_mask']
    for t in (ids, mask):
        assert t.dtype == torch.int64 and t.device == device and tuple(t.shape) == (len(want), width)
    if overflow:
        smp = out['overflow_to_sample_mapping']
        assert smp.dtype == torch.int64 and smp.device == device and smp.cpu().tolist() == want_rows
    else:
        assert 'overflow_to_sample_mapping' not in out
    ids, mask = ids.cpu().numpy(), mask.cpu().numpy()
    lens = np.array([len(w) for w in want], dtype=np.int64)
    j = np.arange(width)[None, :]
    want_mask = (j >= (width - lens)[:, None]) if pad_left else (j < lens[:, None])
    assert np.array_equal(mask, want_mask.astype(np.int64))
    assert np.all(ids[~want_mask] == pad_id)
    flat = np.concatenate([np.asarray(w, dtype=np.int64) for w in want]) if want else np.zeros(0, np.int64)
    assert np.array_equal(ids[want_mask], flat)


def pair_kwargs(strategy, ml, stride, left, pname='longest,right,0', overflow=True):
    mode, pad_left, mult = parse_pad(pname)
    return dict(max_length=ml, padding=mode, truncation=strategy if ml is not None else False, stride=stride,
                return_overflowing_tokens=overflow and ml is not None, pad_to_multiple_of=mult,
                padding_side='left' if pad_left else 'right', truncation_side='left' if left else 'right')


def side_ids(torch, enc_values, enc_splits, rows, dtype, device):
    """the encoder rows `rows` next to each other as (values, splits) on the device"""
    sp = enc_splits.cpu().numpy()
    vals = enc_values.cpu().numpy()
    parts = [vals[sp[r]:sp[r + 1]] for r in rows]
    lens = np.array([len(p) for p in parts], dtype=np.int64)
    v = np.concatenate(parts) if parts else np.zeros(0, np.int32)
    v = torch.from_numpy(v.astype(np.uint16).view(np.int16) if dtype == 'uint16' else v.astype(np.int32))
    return v.to(device), torch.from_numpy(np.concatenate([[0], np.cumsum(lens)])).to(device)


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', ['int32', 'uint16'])
@pytest.mark.parametrize('variant', VARIANTS)
def test_pair_windows_equal_hf(A, fix, golden, content, toks, variant, dtype):
    """Engine.windows_batch(ids, pair_ids=...) on encode_bpe_batch(norm), every strategy, configuration and batch; padded
    widths for the padding subset; a batch with a refused pair raises ValueError"""
    import torch
    V = fix['variants'][variant]
    eng = toks[variant]._eng
    enc = eng.encode_bpe_batch([r['norm'] for r in golden['rows']])
    P = n_template(V)
    sides = []
    for b0, b1 in batches(fix):
        pa = side_ids(torch, enc.values, enc.splits, [a for a, _ in fix['pairs'][b0:b1]], dtype, eng.device)
        pb = side_ids(torch, enc.values, enc.splits, [b for _, b in fix['pairs'][b0:b1]], dtype, eng.device)
        sides.append((pa, pb))
    for strategy in fix['strategies']:
        for name in fix['trunc']:
            ml, stride, left = parse_trunc(name, P)
            for bi, (b0, b1) in enumerate(batches(fix)):
                pa, pb = sides[bi]
                kw = pair_kwargs(strategy, ml, stride, left)
                if batch_refused(V, strategy, name, b0, b1):
                    with pytest.raises(ValueError):
                        eng.windows_batch(pa, 0, pair_ids=pb, **kw)
                    continue
                out = eng.windows_batch(pa, 0, pair_ids=pb, **kw)
                want, want_rows = fixture_windows(V, fix, content, strategy, name, b0, b1)
                check_dense(out, want, want_rows, max(len(w) for w in want), False, 0, eng.device, ml is not None)
                if ml is not None and bi == 0:              # without return_overflowing_tokens: window (0, 0) of every pair
                    out = eng.windows_batch(pa, 0, pair_ids=pb, **pair_kwargs(strategy, ml, stride, left, overflow=False))
                    want, want_rows = fixture_windows(V, fix, content, strategy, name, b0, b1, overflow=False)
                    check_dense(out, want, want_rows, max(len(w) for w in want), False, 0, eng.device, overflow=False)
        for name in fix['pad_trunc']:
            ml, stride, left = parse_trunc(name, P)
            for pname, widths in V['width'][strategy][name].items():
                for bi, (b0, b1) in enumerate(batches(fix)):
                    if widths[bi] is None:
                        continue
                    pa, pb = sides[bi]
                    out = eng.windows_batch(pa, 0, pair_ids=pb, **pair_kwargs(strategy, ml, stride, left, pname))
                    want, want_rows = fixture_windows(V, fix, content, strategy, name, b0, b1)
                    check_dense(out, want, want_rows, widths[bi], parse_pad(pname)[1], 0, eng.device, ml is not None)


@pytest.mark.gpu
@pytest.mark.parametrize('variant', VARIANTS)
def test_encode_batch_tensors_pairs_equal_hf(A, fix, golden, content, toks, variant):
    """aksharTokenizer.encode_batch_tensors(texts, text_pair=...) on the raw `in` strings, against the fixture; the
    transformers batches verbatim"""
    V = fix['variants'][variant]
    tk = toks[variant]
    rows = golden['rows']
    P = n_template(V)
    for strategy in fix['strategies']:
        for name in fix['trunc']:
            ml, stride, left = parse_trunc(name, P)
            for b0, b1 in batches(fix):
                ta = [rows[a]['in'] for a, _ in fix['pairs'][b0:b1]]
                tb = [rows[b]['in'] for _, b in fix['pairs'][b0:b1]]
                kw = pair_kwargs(strategy, ml, stride, left)
                if batch_refused(V, strategy, name, b0, b1):
                    with pytest.raises(ValueError):
                        tk.encode_batch_tensors(ta, text_pair=tb, **kw)
                    continue
                out = tk.encode_batch_tensors(ta, text_pair=tb, **kw)
                want, want_rows = fixture_windows(V, fix, content, strategy, name, b0, b1)
                check_dense(out, want, want_rows, max(len(w) for w in want), False, 0, tk._eng.device, ml is not None)
    for rec in V['verbatim']:
        ml, stride, left = parse_trunc(rec['trunc'], 4)
        b0, b1 = batches(fix)[rec['batch']]
        out = tk.encode_batch_tensors([rows[a]['in'] for a, _ in fix['pairs'][b0:b1]], text_pair=[rows[b]['in'] for _, b in fix['pairs'][b0:b1]],
                                      max_length=ml, stride=stride, truncation=rec['strategy'], return_overflowing_tokens=True,
                                      padding=rec['padding'], truncation_side='left' if left else 'right')
        assert out['input_ids'].tolist() == rec['input_ids']
        assert out['attention_mask'].tolist() == rec['attention_mask']
        assert out['overflow_to_sample_mapping'].tolist() == rec['overflow_to_sample_mapping']


@pytest.mark.gpu
@pytest.mark.parametrize('model,key', [('spm24k.model', 'ids_spm24k'), ('spm_corpus.model', 'ids_spm_corpus')])
def test_unigram_pairs_equal_oracle(A, fix, golden, model, key):
    """the fixture's pairs and configurations on the SentencePiece models (no template ids at all, explicit pad_id)"""
    tk = A.aksharTokenizer(os.path.join(MODELS, model), 'sentencepiece')
    rows = golden['rows']
    enc = tk._eng.encode_unigram_batch([r['norm'] for r in rows])
    import torch
    for strategy in fix['strategies']:
        for name in fix['trunc']:
            ml, stride, left = parse_trunc(name, 0)
            for pname in ('longest,left,8', 'max_length,right,0'):
                if ml is None and pname.startswith('max_length'):
                    continue
                mode, pad_left, mult = parse_pad(pname)
                b0, b1 = batches(fix)[(len(name) + len(strategy)) % 10]
                pa = side_ids(torch, enc.values, enc.splits, [a for a, _ in fix['pairs'][b0:b1]], 'int32', tk._eng.device)
                pb = side_ids(torch, enc.values, enc.splits, [b for _, b in fix['pairs'][b0:b1]], 'int32', tk._eng.device)
                kw = pair_kwargs(strategy, ml, stride, left, pname)
                try:
                    ids, mask, sample = pair_windows([rows[a][key] for a, _ in fix['pairs'][b0:b1]],
                                                     [rows[b][key] for _, b in fix['pairs'][b0:b1]], None, None, [], [], [], ml,
                                                     stride, strategy, left, True, mode, mult, pad_left, 7, truncate=ml is not None)
                except ValueError:
                    with pytest.raises(ValueError):
                        tk._eng.windows_batch(pa, 1, pair_ids=pb, pad_id=7, **kw)
                    continue
                out = tk._eng.windows_batch(pa, 1, pair_ids=pb, pad_id=7, **kw)
                assert out['input_ids'].tolist() == ids and out['attention_mask'].tolist() == mask, (model, strategy, name, pname)
                if ml is not None:
                    assert out['overflow_to_sample_mapping'].tolist() == sample


def dense_of(ids, mask, sample, device):
    import torch
    return {'input_ids': torch.tensor(ids, dtype=torch.int64, device=device).reshape(len(ids), -1),
            'attention_mask': torch.tensor(mask, dtype=torch.int64, device=device).reshape(len(ids), -1),
            'overflow_to_sample_mapping': torch.tensor(sample, dtype=torch.int64, device=device)}


@pytest.mark.gpu
def test_pair_edge_batches(A, toks):
    import torch
    tk = toks['bpe24k']
    eng = tk._eng
    dev = eng.device
    empty = (torch.zeros(0, dtype=torch.int32, device=dev), torch.zeros(1, dtype=torch.int64, device=dev))
    out = eng.windows_batch(empty, 0, pair_ids=empty)
    assert tuple(out['input_ids'].shape) == (0, 0)
    out = eng.windows_batch(empty, 0, pair_ids=empty, max_length=16, padding='max_length', truncation='only_second',
                            return_overflowing_tokens=True)
    assert tuple(out['input_ids'].shape) == (0, 16) and out['overflow_to_sample_mapping'].numel() == 0
    out = tk.encode_batch_tensors([], text_pair=[], max_length=8, truncation=True)
    assert tuple(out['input_ids'].shape) == (0, 0)
    one = tk.encode_batch(['namaste duniya'])[0]
    out = tk.encode_batch_tensors(['', 'namaste duniya', ''], text_pair=['', '', 'namaste duniya'], max_length=64, truncation=True,
                                  return_overflowing_tokens=True)
    assert out['input_ids'].tolist() == [[2, 3, 2, 3] + [0] * (len(one) - 2), one + [2, 3], [2, 3] + one]
    assert out['overflow_to_sample_mapping'].tolist() == [0, 1, 2]
    # one question against a multi-MB context: thousands of windows
    import synth_corpus as sc
    ctx = ' '.join(sc.Corpus('hinglish', 7).lines(4 << 20))
    assert len(ctx.encode('utf-8')) > 3 << 20
    q = 'yeh kahan likha hai?'
    ra, rb = tk.encode_batch([q, ctx])
    for strategy, left in (('only_second', False), ('longest_first', True)):
        kw = dict(max_length=384, stride=128, truncation=strategy, return_overflowing_tokens=True, padding='max_length',
                  truncation_side='left' if left else 'right')
        out = tk.encode_batch_tensors([q], text_pair=[ctx], **kw)
        ids, mask, sample = pair_windows([ra], [rb], 2, 3, [2], [3, 2], [3], 384, 128, strategy, left, True, 'max_length', None,
                                         False, 0)
        assert len(ids) > 1000
        want = dense_of(ids, mask, sample, dev)
        assert all(torch.equal(out[k], want[k]) for k in want)
    # longest_first with wa * wb large: two rows of 1500 content ids, 4 ids each per window, step 1
    g = torch.Generator().manual_seed(3)
    ca = torch.randint(4, 24000, (1500,), generator=g, dtype=torch.int32)
    cb = torch.randint(4, 24000, (1500,), generator=g, dtype=torch.int32)
    two = torch.tensor([2], dtype=torch.int32)
    three = torch.tensor([3], dtype=torch.int32)
    va = torch.cat([two, ca, three]).to(dev)
    vb = torch.cat([two, cb, three]).to(dev)
    sp = torch.tensor([0, 1502], dtype=torch.int64, device=dev)
    out = eng.windows_batch((va, sp), 0, pair_ids=(vb, sp), max_length=12, stride=3, truncation=True, return_overflowing_tokens=True)
    w = 1 + (1500 - 4 + 0) // 1
    assert tuple(out['input_ids'].shape) == (w * w, 12)
    spans = pair_spans(1500, 1500, 8, 3, 'longest_first', False, True)
    a0 = torch.tensor([s[0][0] for s in spans], dtype=torch.int64)
    b0 = torch.tensor([s[1][0] for s in spans], dtype=torch.int64)
    k4 = torch.arange(4)
    want = torch.cat([torch.full((len(spans), 1), 2), ca.long()[a0[:, None] + k4], torch.tensor([[3, 2]]).expand(len(spans), 2),
                      cb.long()[b0[:, None] + k4], torch.full((len(spans), 1), 3)], 1)
    assert torch.equal(out['input_ids'].cpu(), want)
    assert bool(out['attention_mask'].all()) and bool((out['overflow_to_sample_mapping'] == 0).all())


@pytest.mark.gpu
def test_pair_refusals_leave_the_engine_usable(A, toks, tmp_path):
    import torch
    tk = toks['bpe24k']
    eng = tk._eng
    texts = ['yeh ek lambi si line hai jo kai tokens mein tootegi, bilkul', 'chhoti']
    pairs = ['doosri line bhi kaafi lambi hai taaki dono kat jaayen', 'haan']
    ids, _ = tk.encode_batch(texts + pairs, as_device=True)
    a, b = (ids.values, ids.splits[:3]), (ids.values, ids.splits[2:])
    good = dict(max_length=12, truncation=True, stride=1, return_overflowing_tokens=True)
    ref = eng.windows_batch(a, 0, pair_ids=b, **good)
    bad = [dict(max_length=4, truncation=True),                                            # m = max_length - 4 <= 0
           dict(max_length=5, truncation=True),                                            # longest_first cuts a side to 0 ids
           dict(max_length=8, truncation=True, stride=2),                                  # stride >= the cut length
           dict(max_length=12, truncation='only_first', stride=0),                         # A cannot give up enough ids
           dict(max_length=12, truncation='middle'), dict(max_length=12, truncation='only_third'),
           dict(stride=1), dict(return_overflowing_tokens=True),                           # without truncation
           dict(max_length=8, truncation='do_not_truncate', stride=1),
           dict(padding='max_length'),                                                     # no max_length
           dict(max_length=8, padding='max_length')]                                       # a pair longer than L
    for kw in bad:
        with pytest.raises(ValueError):
            eng.windows_batch(a, 0, pair_ids=b, **kw)
        out = eng.windows_batch(a, 0, pair_ids=b, **good)
        assert all(torch.equal(out[k], ref[k]) for k in ref)
    with pytest.raises(ValueError, match='pair 0'):
        eng.windows_batch(a, 0, pair_ids=b, max_length=8, truncation=True, stride=2)
    with pytest.raises(ValueError):                     # rows the encoder did not produce: the template is missing
        eng.windows_batch(a, 0, pair_ids=(ids.values, ids.splits[2:] + torch.tensor([1, 0, 0], device=eng.device)))
    with pytest.raises(ValueError):                     # not the same number of rows
        eng.windows_batch(a, 0, pair_ids=(ids.values, ids.splits[1:]))
    with pytest.raises(ValueError):
        tk.encode_batch_tensors(texts, text_pair=pairs[:1])
    # more than 2^31 - 1 windows
    big = torch.cat([torch.tensor([2]), torch.full((70000,), 7), torch.tensor([3])]).to(torch.int32).to(eng.device)
    sp = torch.tensor([0, 70002], dtype=torch.int64, device=eng.device)
    with pytest.raises(ValueError, match='2\\^31'):
        eng.windows_batch((big, sp), 0, pair_ids=(big, sp), max_length=6, truncation=True, return_overflowing_tokens=True)
    tu = A.aksharTokenizer(os.path.join(MODELS, 'spm24k.model'), 'sentencepiece')
    with pytest.raises(ValueError):                     # no pad piece and no pad_id
        tu.encode_batch_tensors(texts, text_pair=pairs)
    assert tu.encode_batch_tensors(texts, text_pair=pairs, pad_id=0)['input_ids'].shape[0] == 2
    # a pair template of another shape: the model loads and works, pair calls are refused
    j = variant_json('bpe24k')
    j['post_processor']['pair'] = [{'Sequence': {'id': 'B', 'type_id': 0}}, {'Sequence': {'id': 'A', 'type_id': 0}}]
    p = tmp_path / 'odd_pair.json'
    p.write_text(json.dumps(j), encoding='utf-8')
    odd = A.aksharTokenizer(str(p), 'bpe')
    assert odd.encode_batch(texts) == tk.encode_batch(texts)
    assert torch.equal(odd.encode_batch_tensors(texts, max_length=8, truncation=True)['input_ids'],
                       tk.encode_batch_tensors(texts, max_length=8, truncation=True)['input_ids'])
    with pytest.raises(ValueError, match='unsupported pair template'):
        odd.encode_batch_tensors(texts, text_pair=pairs)
    out = eng.windows_batch(a, 0, pair_ids=b, **good)
    assert all(torch.equal(out[k], ref[k]) for k in ref)


# ------------------------------------------------------------------ GPU, at scale
def pair_checksums(values, sa, sb, pre, mid, post, ml, stride, strategy, left, width):
    """per-window sum of id * (position + 1) and sum of mask * (position + 1) of the oracle's layout (right padding),
    from the oracle's spans and prefix sums of the ragged ids; sa / sb: splits of the two sides (rows framed by 2 / 3)"""
    v = values.astype(np.int64)
    p1 = np.concatenate([[0], np.cumsum(v)])
    p2 = np.concatenate([[0], np.cumsum(v * np.arange(v.size))])
    P = len(pre) + len(mid) + len(post)
    ga, la, gb, lb, rows = [], [], [], [], []
    for r in range(sa.size - 1):
        ca, cb = int(sa[r + 1] - sa[r]) - 2, int(sb[r + 1] - sb[r]) - 2
        for (a0, a1), (b0, b1) in pair_spans(ca, cb, ml - P, stride, strategy, left, True):
            ga.append(int(sa[r]) + 1 + a0)
            la.append(a1 - a0)
            gb.append(int(sb[r]) + 1 + b0)
            lb.append(b1 - b0)
            rows.append(r)
    ga, la, gb, lb = (np.array(x, dtype=np.int64) for x in (ga, la, gb, lb))

    def seg(g, n, q0):                                  # ids g .. g + n - 1 at output positions q0 ..
        return (p2[g + n] - p2[g]) + (q0 + 1 - g) * (p1[g + n] - p1[g])
    qa = len(pre)
    qb = qa + la + len(mid)
    ck = seg(ga, la, np.full_like(la, qa)) + seg(gb, lb, qb)
    ck += sum(t * (q + 1) for q, t in enumerate(pre))
    ck += sum(t * (qa + la + q + 1) for q, t in enumerate(mid))
    ck += sum(t * (qb + lb + q + 1) for q, t in enumerate(post))
    tot = la + lb + P
    mk = (1 + tot) * tot // 2
    return ck, mk, np.array(rows, dtype=np.int64)


@pytest.mark.gpu
def test_pairs_at_64mb_equal_oracle(A):
    """rows of 64 MB of Hinglish paired with the rows of the other half, against the oracle's checksums"""
    import torch
    import synth_corpus as sc
    tk = A.aksharTokenizer(os.path.join(MODELS, 'bpe24k.json'), 'bpe')
    eng = tk._eng
    data, off = sc.Corpus('hinglish', 64).generate(64 << 20)
    enc, _ = eng.tokenizer_encode_batch((torch.from_numpy(data), torch.from_numpy(off)), 0)
    h = (enc.splits.numel() - 1) // 2
    sa, sb = enc.splits[:h + 1], enc.splits[h:2 * h + 1]
    values = enc.values.cpu().numpy()
    for strategy, ml, stride, left in (('longest_first', 24, 3, False), ('only_second', 256, 31, True), ('longest_first', 64, 0, True)):
        kw = dict(max_length=ml, truncation=strategy, stride=stride, return_overflowing_tokens=True, padding='max_length',
                  truncation_side='left' if left else 'right')
        sa_np, sb_np = sa.cpu().numpy(), sb.cpu().numpy()
        try:
            ck, mk, rows = pair_checksums(values, sa_np, sb_np, [2], [3, 2], [3], ml, stride, strategy, left, ml)
        except ValueError:
            with pytest.raises(ValueError):
                eng.windows_batch((enc.values, sa), 0, pair_ids=(enc.values, sb), **kw)
            continue
        out = eng.windows_batch((enc.values, sa), 0, pair_ids=(enc.values, sb), **kw)
        w = torch.arange(1, ml + 1, device=eng.device, dtype=torch.int64)
        assert np.array_equal(out['overflow_to_sample_mapping'].cpu().numpy(), rows)
        assert np.array_equal((out['attention_mask'] * w).sum(1).cpu().numpy(), mk)
        assert np.array_equal((out['input_ids'] * w).sum(1).cpu().numpy(), ck), (strategy, ml, stride, left)


@pytest.mark.gpu
def test_pairs_at_1gib_qa_shape(A):
    """1 GiB of Hinglish in the shape of extractive QA: a short row (question) against every document of 512 rows
    (context), only_second, max_length 384, stride 128: the question is whole in every window, the context windows with
    their stride overlap removed give back the context ids, and two halves windowed apart equal the whole"""
    import torch
    import synth_corpus as sc
    tk = A.aksharTokenizer(os.path.join(MODELS, 'bpe24k.json'), 'bpe')
    eng = tk._eng
    dev = eng.device
    data, off = sc.Corpus('hinglish', 20261018).generate(1 << 30)
    enc, _ = eng.tokenizer_encode_batch((torch.from_numpy(data), torch.from_numpy(off)), 0)
    del data, off
    n_rows = enc.splits.numel() - 1
    docs = torch.cat([enc.splits[::512], enc.splits[-1:]]) if n_rows % 512 else enc.splits[::512]
    n_docs = docs.numel() - 1
    lens = enc.splits[1:] - enc.splits[:-1]
    short = torch.nonzero(lens <= 66).flatten()
    q = short[torch.arange(n_docs, device=dev) % short.numel()]
    qs = torch.stack([enc.splits[q], enc.splits[q + 1]], 1)             # one question row per document
    ml, stride = 384, 128
    kw = dict(max_length=ml, truncation='only_second', stride=stride, return_overflowing_tokens=True, padding='max_length')
    # the question rows as a ragged side of their own: their ids gathered next to each other
    qlen = qs[:, 1] - qs[:, 0]
    qsplits = torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), torch.cumsum(qlen, 0)])
    qpos = torch.repeat_interleave(qs[:, 0] - qsplits[:-1], qlen) + torch.arange(int(qsplits[-1]), device=dev)
    qvals = enc.values[qpos]
    out = eng.windows_batch((qvals, qsplits), 0, pair_ids=(enc.values, docs), **kw)
    ids, mask, smp = out['input_ids'], out['attention_mask'], out['overflow_to_sample_mapping']
    ca = (qlen - 2)[smp]
    j = torch.arange(ml, device=dev)[None, :]
    # the question: positions 1 .. ca of every window
    inq = (j >= 1) & (j < 1 + ca[:, None])
    src = (qs[smp, 0] + 1)[:, None] + (j - 1)
    assert torch.equal(ids[inq], enc.values[src[inq]].to(torch.int64))
    del inq, src
    # the context: after <s> A </s> <s>, past the stride overlap for every window but a pair's first
    lb = mask.sum(1) - 4 - ca
    later = torch.cat([torch.zeros(1, dtype=torch.bool, device=dev), smp[1:] == smp[:-1]])
    b0 = 3 + ca + later.to(torch.int64) * stride
    keep = (j >= b0[:, None]) & (j < (3 + ca + lb)[:, None])
    got = ids[keep]
    tmpl = torch.zeros(enc.values.numel(), dtype=torch.bool, device=dev)
    tmpl[docs[:-1]] = True
    tmpl[docs[1:] - 1] = True
    assert torch.equal(got, enc.values[~tmpl].to(torch.int64))
    del got, keep, tmpl
    half = n_docs // 2
    qh = int(qsplits[half])
    a = eng.windows_batch((qvals, qsplits[:half + 1]), 0, pair_ids=(enc.values, docs[:half + 1]), **kw)
    b = eng.windows_batch((qvals[qh:], qsplits[half:] - qh), 0, pair_ids=(enc.values, docs[half:]), **kw)
    assert torch.equal(torch.cat([a['input_ids'], b['input_ids']]), ids)
    assert torch.equal(torch.cat([a['attention_mask'], b['attention_mask']]), mask)
    assert torch.equal(torch.cat([a['overflow_to_sample_mapping'], b['overflow_to_sample_mapping'] + half]), smp)


# ------------------------------------------------------------------ call-level bounds
def stride_probe_cases(fix, variant):
    """(max_length, stride, HF refuses the stride, the pair template leaves no room) for the recorded stride probe"""
    V = fix['variants'][variant]
    return [(ml, st, ref, ml - n_template(V) <= 0) for (ml, st), ref in zip(fix['stride_probe'], V['stride_refused'])]


@pytest.mark.parametrize('variant', VARIANTS)
def test_oracle_stride_bound_equals_hf(fix, variant):
    """a stride above max_length less the single template's ids is refused for the whole call, as HF's enable_truncation
    refuses it, also when no pair is cut"""
    V = fix['variants'][variant]
    bos, eos = (2, 3) if V['template'] else (None, None)
    frame = (lambda c: [2] + c + [3]) if V['template'] else (lambda c: c)
    assert any(ref for _, _, ref, _ in stride_probe_cases(fix, variant))
    for ml, st, ref, no_room in stride_probe_cases(fix, variant):
        args = ([frame([5])], [frame([6])], bos, eos, V['pre'], V['mid'], V['post'], ml, st, 'only_second', False, True, 'longest',
                None, False, 0)
        if ref or no_room:
            with pytest.raises(ValueError, match='stride' if ref and not no_room else ''):
                pair_windows(*args)
        else:
            ids, _, _ = pair_windows(*args)
            assert ids == [V['pre'] + [5] + V['mid'] + [6] + V['post']]


@pytest.mark.gpu
@pytest.mark.parametrize('variant', VARIANTS)
def test_stride_bound_equals_hf(A, fix, toks, variant):
    """the recorded stride probe on a pair of one id a side (never cut), on the device"""
    import torch
    V = fix['variants'][variant]
    eng = toks[variant]._eng
    frame = (lambda c: [2] + c + [3]) if V['template'] else (lambda c: c)
    ra, rb = frame([5]), frame([6])
    a = (torch.tensor(ra, dtype=torch.int32, device=eng.device), torch.tensor([0, len(ra)], dtype=torch.int64, device=eng.device))
    b = (torch.tensor(rb, dtype=torch.int32, device=eng.device), torch.tensor([0, len(rb)], dtype=torch.int64, device=eng.device))
    for ml, st, ref, no_room in stride_probe_cases(fix, variant):
        kw = dict(max_length=ml, stride=st, truncation='only_second', return_overflowing_tokens=True)
        if ref or no_room:
            with pytest.raises(ValueError):
                eng.windows_batch(a, 0, pair_ids=b, **kw)
            continue
        out = eng.windows_batch(a, 0, pair_ids=b, **kw)
        assert out['input_ids'].tolist() == [V['pre'] + [5] + V['mid'] + [6] + V['post']]
        assert out['overflow_to_sample_mapping'].tolist() == [0]


@pytest.mark.gpu
def test_call_window_total_is_bounded(A, toks):
    """pairs that each stay under 2^31 - 1 windows but exceed it together are refused before anything is allocated
    (the window splits are scanned in 32-bit tile sums); the engine gives the same result afterwards"""
    import torch
    tk = toks['bpe24k']
    eng = tk._eng
    dev = eng.device
    g = torch.Generator().manual_seed(5)
    c = 38000                                           # longest_first, max_length 6: both sides cut to 1 id, c * c windows
    assert c * c < 2 ** 31 - 1
    texts, pairs = ['yeh ek lambi si line hai jo kai tokens mein tootegi'], ['doosri line']
    ref = tk.encode_batch_tensors(texts, text_pair=pairs, max_length=8, truncation=True, stride=1, return_overflowing_tokens=True)
    for n_pairs in (2, 3):
        rows = [torch.cat([torch.tensor([2]), torch.randint(4, 24000, (c,), generator=g), torch.tensor([3])]) for _ in range(2 * n_pairs)]
        values = torch.cat(rows).to(torch.int32).to(dev)
        splits = torch.arange(0, 2 * n_pairs + 1, dtype=torch.int64, device=dev) * (c + 2)
        with pytest.raises(ValueError, match='in all'):
            eng.windows_batch((values, splits[:n_pairs + 1]), 0, pair_ids=(values, splits[n_pairs:]), max_length=6, truncation=True,
                              return_overflowing_tokens=True)
        out = tk.encode_batch_tensors(texts, text_pair=pairs, max_length=8, truncation=True, stride=1, return_overflowing_tokens=True)
        assert all(torch.equal(out[k], ref[k]) for k in ref)
    # a refused pair is still named first when the call's total is also too large
    rows = [torch.tensor([2, 5, 3])] + [torch.cat([torch.tensor([2]), torch.randint(4, 24000, (c,), generator=g), torch.tensor([3])])
                                        for _ in range(5)]
    values = torch.cat(rows).to(torch.int32).to(dev)
    splits = torch.tensor([0, 3, 3 + (c + 2), 3 + 2 * (c + 2), 3 + 3 * (c + 2), 3 + 4 * (c + 2), 3 + 5 * (c + 2)], device=dev)
    with pytest.raises(ValueError, match='pair 0'):
        eng.windows_batch((values, splits[:4]), 0, pair_ids=(values, splits[3:]), max_length=6, truncation='only_first',
                          return_overflowing_tokens=True)


@pytest.mark.gpu
def test_mixed_int32_and_compact_sides(A, toks):
    """one side int32, the other compact (uint16 bit patterns in an int16 tensor, ids of 2^15 and above included): the same
    windows as two int32 sides"""
    import torch
    eng = toks['bpe24k']._eng
    dev = eng.device
    a = np.array([2, 40000, 65535, 32768, 5, 3], dtype=np.int64)
    b = np.array([2, 33000, 7, 65000, 3], dtype=np.int64)
    sa = torch.tensor([0, 6], dtype=torch.int64)
    sb = torch.tensor([0, 5], dtype=torch.int64)
    kw = dict(max_length=8, truncation=True, stride=1, return_overflowing_tokens=True)
    i32 = lambda x: torch.from_numpy(x.astype(np.int32))                       # noqa: E731
    c16 = lambda x: torch.from_numpy(x.astype(np.uint16).view(np.int16))       # noqa: E731
    want = eng.windows_batch((i32(a), sa), 0, pair_ids=(i32(b), sb), **kw)
    assert want['input_ids'].tolist()[0] == [2, 40000, 65535, 3, 2, 33000, 7, 3]
    for va, vb in ((i32(a), c16(b)), (c16(a), i32(b)), (c16(a), c16(b))):
        got = eng.windows_batch((va.to(dev), sa), 0, pair_ids=(vb.to(dev), sb), **kw)
        assert all(torch.equal(got[k], want[k]) for k in want)
