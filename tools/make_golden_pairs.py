#!/usr/bin/env python
"""Golden vectors for the model-ready sentence-pair windows (pair template, longest_first / only_first / only_second
truncation with stride, padding), recorded from HF `tokenizers` and `transformers` (their versions are stored as `pins`):
python tools/make_golden_pairs.py -> tests/golden/pairs_hf.json.gz.

Pairs are seeded pairs of the golden rows' `norm` strings in batches of 64: 8 batches drawn from all rows and 2 in the
shape of extractive QA (a short first text, a long second one).  Three variants of bpe24k.json: its own pair template
`<s> $A </s> <s> $B </s>`, the RoBERTa-style `<s> $A </s> </s> $B </s>`, and no post-processor.  Per strategy and
truncation configuration every pair is encoded alone; every window HF returns (the encoding and its `overflowing`, in
that order) is stored as (startA, lenA, startB, lenB) in the pair's untruncated contents (the rows' ids without template
ids, which reference_vectors.json.gz holds), and the script asserts that HF's ids are exactly
pre + A slice + mid + B slice + post.  A pair HF refuses or gets wrong is stored as a kind instead: 'too_short' (HF
raises), 'panic' (stride >= the cut length) or 'wider' (a window longer than max_length).  Each batch is also encoded as
one call without parallelism, and the kind of its error (that of its first refused pair) is stored.  Which
(max_length, stride) HF's enable_truncation refuses outright is stored as `stride_refused`.  For a subset of the configurations the padded width of every batch is
stored, after asserting that HF's padded ids and mask are the layout of tools/windows_oracle.py; two batches are kept
verbatim from transformers' PreTrainedTokenizerFast."""
import contextlib
import gzip
import json
import os
import random
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'tools'))
MODELS = os.path.join(ROOT, 'tests', 'golden', 'models')
BATCH = 64
SEED = 20261020
# (max_length, stride, direction); 'P+k' = the pair template's ids + k, None = truncation off
TRUNC = [(None, 0, 'right'), ('P+1', 0, 'right'), ('P+2', 1, 'left'), ('P+3', 1, 'right'), (8, 2, 'left'), (12, 0, 'right'),
         (16, 3, 'right'), (16, 6, 'left'), (24, 0, 'left'), (32, 7, 'right'), (48, 12, 'left'), (64, 31, 'right'),
         (128, 64, 'left'), (256, 100, 'right'), (384, 128, 'right'), (512, 0, 'left')]
STRATEGIES = ['longest_first', 'only_first', 'only_second']
PAD = [(mode, side, mult) for mode in ('longest', 'max_length') for side in ('right', 'left') for mult in (None, 8)]
PAD_TRUNC = [(None, 0, 'right'), (16, 3, 'right'), (48, 12, 'left'), (384, 128, 'right')]
VARIANTS = [('bpe24k', 'own'), ('bpe24k_roberta', 'roberta'), ('bpe24k_no_template', None)]
# (max_length, stride) around HF's check of the stride against max_length less the single template's ids
STRIDE_PROBE = [(512, 600), (512, 511), (512, 510), (8, 6), (8, 5), (6, 5), (6, 4), (2, 1), (2, 0)]
VERBATIM = [('longest_first', (16, 3, 'right'), 1, 'max_length'), ('only_second', (48, 12, 'left'), 8, 'longest')]


def trunc_name(t):
    return 'none' if t[0] is None else '%s,%d,%s' % t


def pad_name(p):
    return '%s,%s,%s' % (p[0], p[1], p[2] or 0)


def template_json(kind):
    """the post_processor of a variant (None: removed)"""
    if kind is None:
        return None
    j = json.load(open(os.path.join(MODELS, 'bpe24k.json'), encoding='utf-8'))['post_processor']
    if kind == 'roberta':
        s, e = {'SpecialToken': {'id': '<s>', 'type_id': 0}}, {'SpecialToken': {'id': '</s>', 'type_id': 0}}
        j['pair'] = [s, {'Sequence': {'id': 'A', 'type_id': 0}}, e, e, {'Sequence': {'id': 'B', 'type_id': 0}}, e]
    return j


def slots(kind):
    """(pre, mid, post) ids of a variant's pair template"""
    return {'own': ([2], [3, 2], [3]), 'roberta': ([2], [3, 3], [3]), None: ([], [], [])}[kind]


def pairs():
    """(a, b) row indices: 8 batches of any two rows, 2 of a short first row (<= 16 content ids) and a long second one
    (>= 40, the two longest rows included)"""
    with gzip.open(os.path.join(ROOT, 'tests', 'golden', 'reference_vectors.json.gz'), 'rb') as f:
        rows = json.loads(f.read().decode('utf-8'))['rows']
    rng = random.Random(SEED)
    n = len(rows)
    c = [len(r['ids_bpe24k']) - 2 for r in rows]
    out = [(rng.randrange(n), rng.randrange(n)) for _ in range(8 * BATCH)]
    short = [i for i in range(n) if c[i] <= 16]
    long_ = [i for i in range(n) if c[i] >= 40]
    top = sorted(range(n), key=lambda i: -c[i])[:2]
    qa = [(rng.choice(short), rng.choice(long_)) for _ in range(2 * BATCH)]
    qa[5], qa[BATCH + 9] = (qa[5][0], top[0]), (qa[BATCH + 9][0], top[1])
    return rows, out + qa


@contextlib.contextmanager
def quiet_stderr():
    """HF prints a backtrace for every panic; keep the log readable"""
    sys.stderr.flush()
    saved = os.dup(2)
    null = os.open(os.devnull, os.O_WRONLY)
    os.dup2(null, 2)
    try:
        yield
    finally:
        os.dup2(saved, 2)
        os.close(null)
        os.close(saved)


def error_kind(exc):
    if type(exc).__name__ == 'PanicException':
        return 'panic'
    if 'too short' in str(exc):
        return 'too_short'
    raise exc


def locate(content, part, want):
    """start of `part` in content: `want` (the rule's start) if the ids match there, else the first match"""
    k = len(part)
    if want is not None and content[want:want + k] == part:
        return want
    for a in range(len(content) - k + 1):
        if content[a:a + k] == part:
            return a
    raise AssertionError('HF window is not a slice of the content')


def main():
    os.environ['TOKENIZERS_PARALLELISM'] = 'false'     # a batch with refused pairs raises for its first one
    import tokenizers
    import transformers
    from windows_oracle import pair_spans, pair_windows
    rows, prs = pairs()
    norm = [r['norm'] for r in rows]
    content = [r['ids_bpe24k'][1:-1] for r in rows]
    batches = [(b, min(b + BATCH, len(prs))) for b in range(0, len(prs), BATCH)]
    out = {'pins': {'tokenizers': tokenizers.__version__, 'transformers': transformers.__version__}, 'batch': BATCH,
           'pairs': prs, 'strategies': STRATEGIES, 'trunc': [trunc_name(t) for t in TRUNC],
           'pad_trunc': [trunc_name(t) for t in PAD_TRUNC], 'pad': [pad_name(p) for p in PAD], 'stride_probe': STRIDE_PROBE,
           'variants': {}}
    for name, kind in VARIANTS:
        j = json.load(open(os.path.join(MODELS, 'bpe24k.json'), encoding='utf-8'))
        j['post_processor'] = template_json(kind)
        tk = tokenizers.Tokenizer.from_str(json.dumps(j))
        pre, mid, post = slots(kind)
        P = len(pre) + len(mid) + len(post)
        tk.no_truncation()
        tk.no_padding()
        bos, eos = ([2], [3]) if kind else ([], [])
        for a, b in prs[:BATCH]:
            assert tk.encode(norm[a], norm[b]).ids == pre + content[a] + mid + content[b] + post
        assert tk.encode(norm[0]).ids == bos + content[0] + eos
        V = {'template': kind, 'pre': pre, 'mid': mid, 'post': post, 'pad_id': 0, 'windows': {}, 'batch_error': {},
             'width': {}, 'verbatim': []}
        for strategy in STRATEGIES:
            W, E = {}, {}
            for t in TRUNC:
                ml = P + int(t[0][2:]) if isinstance(t[0], str) else t[0]
                tk.no_padding()
                if ml is None:
                    tk.no_truncation()
                else:
                    tk.enable_truncation(ml, stride=t[1], strategy=strategy, direction=t[2])
                per = []
                for a, b in prs:
                    try:
                        with quiet_stderr():
                            e = tk.encode(norm[a], norm[b])
                    except BaseException as x:      # noqa: B036 -- PanicException derives from BaseException
                        per.append(error_kind(x))
                        continue
                    wins = [e] + list(e.overflowing)
                    if ml is not None and any(len(w.ids) > ml for w in wins):
                        per.append('wider')
                        continue
                    try:
                        rule = pair_spans(len(content[a]), len(content[b]), None if ml is None else ml - P, t[1], strategy,
                                          t[2] == 'left', True)
                    except ValueError:
                        rule = None
                    flat = []
                    for k, w in enumerate(wins):
                        ids = w.ids
                        assert ids[:len(pre)] == pre and ids[len(ids) - len(post):] == post
                        inner = ids[len(pre):len(ids) - len(post)]
                        want = rule[k] if rule and k < len(rule) else None
                        # how HF's ids split into A and B where more than one split fits (the ids are the same either
                        # way): the rule's, else HF's sequence ids (not reliable in overflow windows), else any
                        tries = ([want[0][1] - want[0][0]] if want else []) + [w.sequence_ids.count(0)] + list(range(len(inner) + 1))
                        for la in tries:
                            lb = len(inner) - len(mid) - la
                            pa, pb = inner[:la], inner[la + len(mid):]
                            if lb < 0 or inner[la:la + len(mid)] != mid:
                                continue
                            try:
                                sa = locate(content[a], pa, want[0][0] if want else None)
                                sb = locate(content[b], pb, want[1][0] if want else None)
                                break
                            except AssertionError:
                                continue
                        else:
                            raise AssertionError('HF window is not pre + A slice + mid + B slice + post')
                        assert ids == pre + content[a][sa:sa + la] + mid + content[b][sb:sb + lb] + post, (name, strategy, t)
                        flat += [sa, la, sb, lb]
                    per.append(flat)
                W[trunc_name(t)] = per
                errs = []
                for b0, b1 in batches:
                    try:
                        with quiet_stderr():
                            encs = tk.encode_batch([(norm[a], norm[b]) for a, b in prs[b0:b1]])
                        wider = ml is not None and any(len(w.ids) > ml for e in encs for w in [e] + list(e.overflowing))
                        errs.append('wider' if wider else None)
                    except BaseException as x:      # noqa: B036
                        errs.append(error_kind(x))
                E[trunc_name(t)] = errs
                print(name, strategy, trunc_name(t), 'windows', sum(len(x) // 4 for x in per if isinstance(x, list)),
                      'refused', sum(isinstance(x, str) for x in per), flush=True)
            V['windows'][strategy], V['batch_error'][strategy] = W, E
        # padded widths: HF's padded batch is the oracle's layout
        for strategy in STRATEGIES:
            widths = {}
            for t in PAD_TRUNC:
                ml = t[0]
                if ml is None:
                    tk.no_truncation()
                else:
                    tk.enable_truncation(ml, stride=t[1], strategy=strategy, direction=t[2])
                per_pad = {}
                for p in PAD:
                    if p[0] == 'max_length' and ml is None:
                        continue
                    tk.enable_padding(direction=p[1], pad_id=0, pad_token='<pad>', length=ml if p[0] == 'max_length' else None,
                                      pad_to_multiple_of=p[2])
                    ws = []
                    for b0, b1 in batches:
                        ra = [bos + content[a] + eos for a, _ in prs[b0:b1]]
                        rb = [bos + content[b] + eos for _, b in prs[b0:b1]]
                        try:
                            o_ids, o_mask, _ = pair_windows(ra, rb, bos[0] if bos else None, eos[0] if eos else None, pre, mid, post,
                                                            ml, t[1], strategy, t[2] == 'left', True, p[0], p[2], p[1] == 'left', 0,
                                                            truncate=ml is not None)
                        except ValueError:
                            ws.append(None)
                            continue
                        encs = tk.encode_batch([(norm[a], norm[b]) for a, b in prs[b0:b1]])
                        hf_ids = [w.ids for e in encs for w in [e] + list(e.overflowing)]
                        hf_mask = [w.attention_mask for e in encs for w in [e] + list(e.overflowing)]
                        assert hf_ids == o_ids and hf_mask == o_mask, (name, strategy, t, p, b0)
                        ws.append(len(hf_ids[0]))
                    per_pad[pad_name(p)] = ws
                widths[trunc_name(t)] = per_pad
            V['width'][strategy] = widths
        tk.no_padding()
        # which (max_length, stride) HF refuses before encoding anything
        refused = []
        for ml, st in STRIDE_PROBE:
            try:
                tk.enable_truncation(ml, stride=st, strategy='only_second')
                refused.append(False)
            except ValueError:
                refused.append(True)
        V['stride_refused'] = refused
        tk.no_truncation()
        if kind == 'own':
            path = os.path.join(MODELS, 'bpe24k.json')
            ht = transformers.PreTrainedTokenizerFast(tokenizer_file=path, pad_token='<pad>')
            for strategy, t, bi, padding in VERBATIM:
                b0, b1 = batches[bi]
                ht.truncation_side = t[2]
                o = ht([norm[a] for a, _ in prs[b0:b1]], [norm[b] for _, b in prs[b0:b1]], truncation=strategy, max_length=t[0],
                       stride=t[1], return_overflowing_tokens=True, padding=padding)
                V['verbatim'].append({'strategy': strategy, 'trunc': trunc_name(t), 'batch': bi, 'padding': padding,
                                      'input_ids': o['input_ids'], 'attention_mask': o['attention_mask'],
                                      'overflow_to_sample_mapping': o['overflow_to_sample_mapping']})
        out['variants'][name] = V
    path = os.path.join(ROOT, 'tests', 'golden', 'pairs_hf.json.gz')
    with gzip.GzipFile(path, 'wb', mtime=0) as f:
        f.write(json.dumps(out, separators=(',', ':')).encode('utf-8'))
    print('wrote', path, os.path.getsize(path))


if __name__ == '__main__':
    main()
