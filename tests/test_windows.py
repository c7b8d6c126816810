"""Model-ready windows (truncation, stride windows, padding): the oracle (tools/windows_oracle.py) against what HF
tokenizers returned (tests/golden/windows_hf.json.gz, tools/make_golden_windows.py), and the device path
(Engine.windows_batch, aksharTokenizer.encode_batch_tensors) against both."""
import gzip
import json
import os

import numpy as np
import pytest

from windows_oracle import window_spans, windows

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, 'tests', 'golden')
MODELS = os.path.join(GOLDEN, 'models')
IDS_KEY = {'bpe24k': 'ids_bpe24k', 'bpe_corpus': 'ids_bpe_corpus', 'bpe24k_no_template': 'ids_bpe24k'}


@pytest.fixture(scope='module')
def fix():
    with gzip.open(os.path.join(GOLDEN, 'windows_hf.json.gz'), 'rb') as f:
        return json.loads(f.read().decode('utf-8'))


def parse_trunc(name, s):
    """fixture name -> (max_length or None, stride, left)"""
    if name == 'none':
        return None, 0, False
    ml, st, d = name.split(',')
    return (s + 1 if ml == 's+1' else int(ml)), int(st), d == 'left'


def parse_pad(name):
    mode, side, mult = name.split(',')
    return mode, side == 'left', int(mult) or None


def batches(fix, n):
    b = fix['batch']
    return [(i, min(i + b, n)) for i in range(0, n, b)]


def rows_of(V, golden_rows, key):
    """the encoder rows of a variant: with their template ids, or the content alone"""
    return [r[key] for r in golden_rows] if V['template'] else [r[key][1:-1] for r in golden_rows]


def hf_windows(V, name, content, b0, b1, overflow=True):
    """HF's windows of rows b0..b1-1 (template ids included) and their rows, from the recorded (start, length) pairs"""
    head, tail = ([V['bos']] if V['template'] else []), ([V['eos']] if V['template'] else [])
    out, rows = [], []
    for r in range(b0, b1):
        sp = V['windows'][name][r]
        for k in range(0, len(sp) if overflow else 2, 2):
            out.append(head + content[r][sp[k]:sp[k] + sp[k + 1]] + tail)
            rows.append(r - b0)
    return out, rows


def unpad(ids, mask):
    return [[i for i, m in zip(a, b) if m] for a, b in zip(ids, mask)]


# ------------------------------------------------------------------ CPU: the oracle is HF
def test_fixture_holds_every_configuration(fix):
    assert fix['pins']['tokenizers'] == '0.22.2'
    assert set(fix['variants']) == set(IDS_KEY)
    assert len(fix['trunc']) == 10 and len(fix['pad']) == 8


@pytest.mark.parametrize('variant', sorted(IDS_KEY))
def test_oracle_windows_equal_hf(fix, golden, variant):
    V = fix['variants'][variant]
    rows = rows_of(V, golden['rows'], IDS_KEY[variant])
    content = [r[IDS_KEY[variant]][1:-1] for r in golden['rows']]
    s = 2 if V['template'] else 0
    for name in fix['trunc']:
        ml, stride, left = parse_trunc(name, s)
        for overflow in ((True, False) if ml is not None else (False,)):
            for b0, b1 in batches(fix, len(rows)):
                ids, mask, sample = windows(rows[b0:b1], V['bos'], V['eos'], ml, stride, left, overflow, 'longest', None, False,
                                            0, truncate=ml is not None)
                want, want_rows = hf_windows(V, name, content, b0, b1, overflow)
                assert unpad(ids, mask) == want, (variant, name, b0)
                assert sample == want_rows


@pytest.mark.parametrize('variant', sorted(IDS_KEY))
def test_oracle_width_equals_hf(fix, golden, variant):
    V = fix['variants'][variant]
    rows = rows_of(V, golden['rows'], IDS_KEY[variant])
    s = 2 if V['template'] else 0
    for name in fix['trunc']:
        ml, stride, left = parse_trunc(name, s)
        for pname, widths in V['width'][name].items():
            mode, pad_left, mult = parse_pad(pname)
            for bi, (b0, b1) in enumerate(batches(fix, len(rows))):
                ids, mask, _ = windows(rows[b0:b1], V['bos'], V['eos'], ml, stride, left, True, mode, mult, pad_left, 0,
                                       truncate=ml is not None)
                assert len(ids[0]) == widths[bi], (variant, name, pname, bi)
                assert all(len(x) == widths[bi] for x in ids)


def test_oracle_equals_hf_verbatim(fix, golden):
    V = fix['variants']['bpe24k']
    rows = [r['ids_bpe24k'] for r in golden['rows']]
    assert len(V['verbatim']) == 2
    for rec in V['verbatim']:
        ml, stride, left = parse_trunc(rec['trunc'], 2)
        mode, pad_left, mult = parse_pad(rec['pad'])
        b0, b1 = batches(fix, len(rows))[rec['batch']]
        ids, mask, _ = windows(rows[b0:b1], 2, 3, ml, stride, left, True, mode, mult, pad_left, 0)
        assert ids == rec['input_ids'] and mask == rec['attention_mask']


def test_oracle_refuses_what_hf_gets_wrong():
    rows = [[2, 10, 11, 12, 3]]
    for ml in (1, 2):                                   # max_length <= template ids
        with pytest.raises(ValueError):
            windows(rows, 2, 3, ml, 0, False, True, 'longest', None, False, 0)
    with pytest.raises(ValueError):                     # stride >= max_length - template ids
        windows(rows, 2, 3, 4, 2, False, True, 'longest', None, False, 0)
    with pytest.raises(ValueError):                     # a row longer than max_length without truncation
        windows(rows, 2, 3, 4, 0, False, False, 'max_length', None, False, 0, truncate=False)
    assert window_spans(10, 4, 1, False, True) == [(0, 4), (3, 7), (6, 10)]
    assert window_spans(10, 4, 1, True, True) == [(6, 10), (3, 7), (0, 4)]


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
def toks(A, tmp_path_factory):
    """one tokenizer per fixture variant"""
    j = json.load(open(os.path.join(MODELS, 'bpe24k.json'), encoding='utf-8'))
    j['post_processor'] = None
    p = tmp_path_factory.mktemp('models') / 'bpe24k_no_template.json'
    p.write_text(json.dumps(j), encoding='utf-8')
    return {'bpe24k': A.aksharTokenizer(os.path.join(MODELS, 'bpe24k.json'), 'bpe'),
            'bpe_corpus': A.aksharTokenizer(os.path.join(MODELS, 'bpe_corpus.json'), 'bpe'),
            'bpe24k_no_template': A.aksharTokenizer(str(p), 'bpe')}


def kwargs_of(ml, stride, left, pname, overflow=True):
    mode, pad_left, mult = parse_pad(pname)
    return dict(max_length=ml, padding=mode, truncation=ml is not None, stride=stride, return_overflowing_tokens=overflow and ml is not None,
                pad_to_multiple_of=mult, padding_side='left' if pad_left else 'right', truncation_side='left' if left else 'right')


def check_dense(out, want, want_rows, width, pad_left, pad_id, device, overflow=True):
    """the device tensors hold exactly the windows `want` (lists of ids), padded to `width`"""
    import torch
    ids, mask = out['input_ids'], out['attention_mask']
    for t in (ids, mask):
        assert t.dtype == torch.int64 and t.device == device and tuple(t.shape) == (len(want), width)
    if overflow:
        smp = out['overflow_to_sample_mapping']
        assert smp.dtype == torch.int64 and smp.device == device and smp.cpu().tolist() == want_rows
    ids, mask = ids.cpu().numpy(), mask.cpu().numpy()
    lens = np.array([len(w) for w in want], dtype=np.int64)
    j = np.arange(width)[None, :]
    want_mask = (j >= (width - lens)[:, None]) if pad_left else (j < lens[:, None])
    assert np.array_equal(mask, want_mask.astype(np.int64))
    assert np.all(ids[~want_mask] == pad_id)
    flat = np.concatenate([np.asarray(w, dtype=np.int64) for w in want]) if want else np.zeros(0, np.int64)
    assert np.array_equal(ids[want_mask], flat)


@pytest.mark.gpu
@pytest.mark.parametrize('variant', sorted(IDS_KEY))
def test_windows_batch_equals_hf(A, fix, golden, toks, variant):
    """Engine.windows_batch on encode_bpe_batch(norm), every fixture configuration, batch by batch"""
    from akshar_b200.batch import Ragged
    V = fix['variants'][variant]
    eng = toks[variant]._eng
    rows = golden['rows']
    enc = eng.encode_bpe_batch([r['norm'] for r in rows])
    content = [r[IDS_KEY[variant]][1:-1] for r in rows]
    s = 2 if V['template'] else 0
    for name in fix['trunc']:
        ml, stride, left = parse_trunc(name, s)
        for pname, widths in V['width'][name].items():
            for bi, (b0, b1) in enumerate(batches(fix, len(rows))):
                out = eng.windows_batch(Ragged(enc.values, enc.splits[b0:b1 + 1]), 0, **kwargs_of(ml, stride, left, pname))
                want, want_rows = hf_windows(V, name, content, b0, b1)
                check_dense(out, want, want_rows, widths[bi], parse_pad(pname)[1], 0, eng.device, ml is not None)
        if ml is not None:                              # without return_overflowing_tokens: window 0 of every row
            b0, b1 = batches(fix, len(rows))[-1]
            out = eng.windows_batch(Ragged(enc.values, enc.splits[b0:b1 + 1]), 0, **kwargs_of(ml, stride, left, 'longest,right,0', False))
            want, want_rows = hf_windows(V, name, content, b0, b1, overflow=False)
            check_dense(out, want, want_rows, max(len(w) for w in want), False, 0, eng.device, overflow=False)
            assert 'overflow_to_sample_mapping' not in out


@pytest.mark.gpu
@pytest.mark.parametrize('variant', sorted(IDS_KEY))
def test_encode_batch_tensors_equals_hf(A, fix, golden, toks, variant):
    """aksharTokenizer.encode_batch_tensors on the raw `in` strings, every fixture configuration, batch by batch"""
    V = fix['variants'][variant]
    tk = toks[variant]
    rows = golden['rows']
    content = [r[IDS_KEY[variant]][1:-1] for r in rows]
    s = 2 if V['template'] else 0
    for name in fix['trunc']:
        ml, stride, left = parse_trunc(name, s)
        for pname, widths in V['width'][name].items():
            for bi, (b0, b1) in enumerate(batches(fix, len(rows))):
                out = tk.encode_batch_tensors([r['in'] for r in rows[b0:b1]], **kwargs_of(ml, stride, left, pname))
                want, want_rows = hf_windows(V, name, content, b0, b1)
                check_dense(out, want, want_rows, widths[bi], parse_pad(pname)[1], 0, tk._eng.device, ml is not None)


def oracle_dense(rows, ml, stride, left, pname, pad_id, overflow=True):
    """the oracle's windows (unpadded) and padded width for rows without template ids"""
    mode, pad_left, mult = parse_pad(pname)
    ids, mask, sample = windows(rows, None, None, ml, stride, left, overflow and ml is not None, mode, mult, pad_left, pad_id,
                                truncate=ml is not None)
    return unpad(ids, mask), sample, (len(ids[0]) if ids else 0)


@pytest.mark.gpu
@pytest.mark.parametrize('model,key', [('spm24k.model', 'ids_spm24k'), ('spm_corpus.model', 'ids_spm_corpus')])
def test_unigram_windows_equal_oracle(A, fix, golden, model, key):
    """the fixture's configurations on the SentencePiece models (no template ids, no pad piece: explicit pad_id), against
    the oracle on the golden rows; covers the 12 207- and 17 001-token rows"""
    from akshar_b200.batch import Ragged
    tk = A.aksharTokenizer(os.path.join(MODELS, model), 'sentencepiece')
    rows = golden['rows']
    enc = tk._eng.encode_unigram_batch([r['norm'] for r in rows])
    want_rows_all = [r[key] for r in rows]
    for name in fix['trunc']:
        ml, stride, left = parse_trunc(name, 0)
        for pname in fix['pad']:
            if ml is None and pname.startswith('max_length'):
                continue
            for b0, b1 in batches(fix, len(rows)):
                want, want_rows, width = oracle_dense(want_rows_all[b0:b1], ml, stride, left, pname, 7)
                out = tk._eng.windows_batch(Ragged(enc.values, enc.splits[b0:b1 + 1]), 1, pad_id=7,
                                            **kwargs_of(ml, stride, left, pname))
                check_dense(out, want, want_rows, width, parse_pad(pname)[1], 7, tk._eng.device, ml is not None)


@pytest.mark.gpu
def test_uint16_ids_equal_int32(A, golden, toks):
    """the compact uint16 ids of the host-link encoder (held in an int16 tensor) give what the int32 ids give, also for ids of
    2^15 and above (negative int16 bit patterns)"""
    import torch
    from akshar_b200.batch import pack_host
    tk = toks['bpe24k']
    eng = tk._eng
    ins = [r['in'] for r in golden['rows']]
    enc, _ = eng.tokenizer_encode_batch(ins, 0)
    data, off = pack_host(ins)
    compact = tk.encode_batch_host(data, off, compact=True)
    assert compact.ids16.dtype == torch.int16
    u16 = (compact.ids16.to(eng.device), torch.from_numpy(compact.row_splits()).to(eng.device))
    kw = dict(max_length=32, truncation=True, stride=7, return_overflowing_tokens=True, padding='max_length', padding_side='left')
    a = eng.windows_batch(enc, 0, **kw)
    b = eng.windows_batch(u16, 0, **kw)
    for k in a:
        assert torch.equal(a[k], b[k])
    wide = np.array([2, 40000, 65535, 32768, 5, 3, 2, 3], dtype=np.int64)
    sp = torch.tensor([0, 6, 8], dtype=torch.int64)
    a = eng.windows_batch((torch.from_numpy(wide.astype(np.int32)), sp), 0, max_length=4, truncation=True, stride=1,
                          return_overflowing_tokens=True)
    b = eng.windows_batch((torch.from_numpy(wide.astype(np.uint16).view(np.int16)), sp), 0, max_length=4, truncation=True,
                          stride=1, return_overflowing_tokens=True)
    for k in a:
        assert torch.equal(a[k], b[k])
    assert a['input_ids'].tolist() == [[2, 40000, 65535, 3], [2, 65535, 32768, 3], [2, 32768, 5, 3], [2, 3, 0, 0]]


@pytest.mark.gpu
def test_edge_batches(A, toks):
    import torch
    tk = toks['bpe24k']
    eng = tk._eng
    dev = eng.device
    empty = (torch.zeros(0, dtype=torch.int32, device=dev), torch.zeros(1, dtype=torch.int64, device=dev))
    out = eng.windows_batch(empty, 0)
    assert tuple(out['input_ids'].shape) == (0, 0)
    out = eng.windows_batch(empty, 0, max_length=16, padding='max_length', truncation=True, return_overflowing_tokens=True)
    assert tuple(out['input_ids'].shape) == (0, 16) and out['overflow_to_sample_mapping'].numel() == 0
    out = tk.encode_batch_tensors(['', '', ''], max_length=8, truncation=True, return_overflowing_tokens=True)
    assert out['input_ids'].tolist() == [[2, 3]] * 3 and out['attention_mask'].tolist() == [[1, 1]] * 3
    assert out['overflow_to_sample_mapping'].tolist() == [0, 1, 2]
    one = tk.encode_batch(['namaste duniya'])[0]
    out = tk.encode_batch_tensors(['namaste duniya'], max_length=len(one) + 3, padding='max_length')
    assert out['input_ids'].tolist() == [one + [0, 0, 0]] and out['attention_mask'].tolist() == [[1] * len(one) + [0, 0, 0]]
    tu = A.aksharTokenizer(os.path.join(MODELS, 'spm24k.model'), 'sentencepiece')
    out = tu.encode_batch_tensors(['', ''], pad_id=0)
    assert tuple(out['input_ids'].shape) == (2, 0)


@pytest.mark.gpu
def test_refusals_leave_the_engine_usable(A, toks):
    import torch
    tk = toks['bpe24k']
    eng = tk._eng
    texts = ['yeh ek lambi si line hai jo kai tokens mein tootegi, bilkul', 'chhoti']
    enc, _ = tk.encode_batch(texts, as_device=True)
    good = dict(max_length=8, truncation=True, stride=2, return_overflowing_tokens=True)
    ref = eng.windows_batch(enc, 0, **good)
    bad = [dict(max_length=2, truncation=True), dict(max_length=1, truncation=True),             # max_length <= template ids
           dict(max_length=8, truncation=True, stride=6), dict(max_length=8, truncation=True, stride=7),   # stride >= m
           dict(padding='max_length'),                                                        # no max_length
           dict(max_length=4, padding='max_length'),                                          # a row longer than L
           dict(stride=1), dict(return_overflowing_tokens=True), dict(max_length=8, stride=1),    # without truncation
           dict(padding='do_not_pad'), dict(max_length=8, truncation=True, truncation_side='middle')]
    for kw in bad:
        with pytest.raises(ValueError):
            eng.windows_batch(enc, 0, **kw)
        out = eng.windows_batch(enc, 0, **good)
        assert all(torch.equal(out[k], ref[k]) for k in ref)
    with pytest.raises(ValueError):                     # ids the encoder did not produce: the template is missing
        eng.windows_batch((enc.values[1:], enc.splits - torch.tensor([0, 1, 1], device=eng.device)), 0)
    tu = A.aksharTokenizer(os.path.join(MODELS, 'spm24k.model'), 'sentencepiece')
    with pytest.raises(ValueError):                     # no pad piece and no pad_id
        tu.encode_batch_tensors(texts)
    assert tu.encode_batch_tensors(texts, pad_id=0)['input_ids'].shape[0] == 2
    with pytest.raises(ValueError):
        A.aksharTokenizer().encode_batch_tensors(texts)
    out = eng.windows_batch(enc, 0, **good)
    assert all(torch.equal(out[k], ref[k]) for k in ref)


# ------------------------------------------------------------------ GPU, at scale
def window_checksums(values, splits, bos, eos, ml, stride, left, width, pad_left):
    """per-window sum of id * (position + 1) and sum of mask * (position + 1) of the oracle's layout (pad_id 0), from the
    oracle's spans and prefix sums of the ragged ids"""
    head, s = int(bos is not None), int(bos is not None) + int(eos is not None)
    v = values.astype(np.int64)
    p1 = np.concatenate([[0], np.cumsum(v)])
    p2 = np.concatenate([[0], np.cumsum(v * np.arange(v.size))])
    g0, ln, rows = [], [], []
    for r in range(splits.size - 1):
        base, c = int(splits[r]) + head, int(splits[r + 1] - splits[r]) - s
        for a, b in window_spans(c, ml - s, stride, left, True):
            g0.append(base + a)
            ln.append(b - a)
            rows.append(r)
    g0, ln = np.array(g0, dtype=np.int64), np.array(ln, dtype=np.int64)
    tot = ln + s
    first = width - tot if pad_left else np.zeros_like(tot)          # output position of the window's first id
    q0 = first + head                                                # of its first content id
    ck = (p2[g0 + ln] - p2[g0]) + (q0 + 1 - g0) * (p1[g0 + ln] - p1[g0])
    if bos is not None:
        ck += bos * (first + 1)
    if eos is not None:
        ck += eos * (q0 + ln + 1)
    mk = (first + 1 + first + tot) * tot // 2
    return ck, mk, np.array(rows, dtype=np.int64)


@pytest.mark.gpu
@pytest.mark.parametrize('kind,corpus,model', [(0, 'hinglish', 'bpe24k.json'), (1, 'hindi', 'spm24k.model')])
def test_windows_at_64mb_equal_oracle(A, kind, corpus, model):
    import torch
    import synth_corpus as sc
    tk = A.aksharTokenizer(os.path.join(MODELS, model), 'bpe' if kind == 0 else 'sentencepiece')
    eng = tk._eng
    data, off = sc.Corpus(corpus, 64).generate(64 << 20)
    enc, _ = eng.tokenizer_encode_batch((torch.from_numpy(data), torch.from_numpy(off)), kind)
    values, splits = enc.values.cpu().numpy(), enc.splits.cpu().numpy()
    bos, eos = (2, 3) if kind == 0 else (None, None)
    for ml, stride, left, pad_left in ((16, 5, False, False), (64, 0, True, True), (128, 31, True, False)):
        out = eng.windows_batch(enc, kind, max_length=ml, truncation=True, stride=stride, return_overflowing_tokens=True,
                                padding='max_length', truncation_side='left' if left else 'right',
                                padding_side='left' if pad_left else 'right', pad_id=0)
        w = torch.arange(1, ml + 1, device=eng.device, dtype=torch.int64)
        got_ck = (out['input_ids'] * w).sum(1).cpu().numpy()
        got_mk = (out['attention_mask'] * w).sum(1).cpu().numpy()
        ck, mk, rows = window_checksums(values, splits, bos, eos, ml, stride, left, ml, pad_left)
        assert np.array_equal(out['overflow_to_sample_mapping'].cpu().numpy(), rows)
        assert np.array_equal(got_mk, mk) and np.array_equal(got_ck, ck), (ml, stride, left)


@pytest.mark.gpu
def test_windows_at_1gib_give_back_the_ids(A):
    """documents of 512 encoded rows of 1 GiB of Hinglish, max_length 512, stride 128: pads, template ids and the stride
    overlap removed on the device give back the ids; N follows the formula; two halves windowed apart equal the whole"""
    import torch
    import synth_corpus as sc
    tk = A.aksharTokenizer(os.path.join(MODELS, 'bpe24k.json'), 'bpe')
    eng = tk._eng
    data, off = sc.Corpus('hinglish', 20261018).generate(1 << 30)
    enc, _ = eng.tokenizer_encode_batch((torch.from_numpy(data), torch.from_numpy(off)), 0)
    del data, off
    n_rows = enc.splits.numel() - 1
    docs = torch.cat([enc.splits[::512], enc.splits[-1:]]) if n_rows % 512 else enc.splits[::512]
    ml, stride = 512, 128
    m, step = ml - 2, ml - 2 - stride
    kw = dict(max_length=ml, truncation=True, stride=stride, return_overflowing_tokens=True, padding='max_length')
    out = eng.windows_batch((enc.values, docs), 0, **kw)
    ids, mask, smp = out['input_ids'], out['attention_mask'], out['overflow_to_sample_mapping']
    c = docs[1:] - docs[:-1] - 2
    n = torch.where(c <= m, torch.ones_like(c), 1 + torch.div(c - m + step - 1, step, rounding_mode='floor'))
    assert int(n.sum()) == ids.shape[0]
    # content positions of every window: after <s>, before </s>, and past the stride overlap for every window but a row's first
    lens = mask.sum(1) - 2
    later = torch.cat([torch.zeros(1, dtype=torch.bool, device=ids.device), smp[1:] == smp[:-1]])
    j = torch.arange(ml, device=ids.device)[None, :]
    keep = (j >= 1 + later[:, None].to(torch.int64) * stride) & (j < 1 + lens[:, None])
    got = ids[keep]
    tmpl = torch.zeros(enc.values.numel(), dtype=torch.bool, device=ids.device)
    tmpl[docs[:-1]] = True
    tmpl[docs[1:] - 1] = True
    assert torch.equal(got, enc.values[~tmpl].to(torch.int64))
    del got, keep, tmpl
    half = (docs.numel() - 1) // 2
    a = eng.windows_batch((enc.values, docs[:half + 1]), 0, **kw)
    b = eng.windows_batch((enc.values, docs[half:]), 0, **kw)
    assert torch.equal(torch.cat([a['input_ids'], b['input_ids']]), ids)
    assert torch.equal(torch.cat([a['attention_mask'], b['attention_mask']]), mask)
    assert torch.equal(torch.cat([a['overflow_to_sample_mapping'], b['overflow_to_sample_mapping'] + half]), smp)
