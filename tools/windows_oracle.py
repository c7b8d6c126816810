"""Plain-Python restatement of the model-ready windowing of HF `tokenizers` (Tokenizer.enable_truncation(max_length,
stride, direction) + enable_padding(direction, pad_id, length, pad_to_multiple_of) + encode_batch, flattened the way
transformers returns `[enc] + enc.overflowing`).  The reference that tests/test_windows.py checks against the recorded HF
results and that the device path (Engine.windows_batch) is compared with.  No torch, no tokenizers."""


def window_spans(n, m, stride, left, overflow):
    """(start, stop) of every window of a row with n content ids (template ids excluded), m = max_length - specials;
    m = None: no truncation (one window)"""
    if m is None or n <= m:
        return [(0, n)]
    step = m - stride
    spans = []
    k = 0
    while True:
        if left:
            stop = n - k * step
            start = max(stop - m, 0)
        else:
            start = k * step
            stop = min(start + m, n)
        spans.append((start, stop))
        if not overflow or (start == 0 if left else stop == n):
            return spans
        k += 1


def windows(rows, bos, eos, max_length, stride, left, overflow, padding, multiple, pad_left, pad_id, truncate=True):
    """rows: encoder output rows (with their template ids); bos / eos: the template's ids or None.
    -> (input_ids [N][L], attention_mask [N][L], overflow_to_sample_mapping [N]) as lists"""
    head, tail = (0 if bos is None else 1), (0 if eos is None else 1)
    s = head + tail
    if truncate and max_length <= s:
        raise ValueError('max_length must exceed the %d template ids' % s)
    m = max_length - s if truncate else None
    if m is not None and stride >= m:
        raise ValueError('stride must be smaller than max_length - template ids')
    out, sample = [], []
    for r, row in enumerate(rows):
        row = list(row)
        c = row[head:len(row) - tail]
        for a, b in window_spans(len(c), m, stride, left, overflow):
            out.append(([bos] if head else []) + c[a:b] + ([eos] if tail else []))
            sample.append(r)
    width = max_length if padding == 'max_length' else max((len(w) for w in out), default=0)
    if multiple:
        width = (width + multiple - 1) // multiple * multiple
    if any(len(w) > width for w in out):
        raise ValueError('a row is longer than the padded width')
    ids, mask = [], []
    for w in out:
        pad = width - len(w)
        ids.append([pad_id] * pad + w if pad_left else w + [pad_id] * pad)
        mask.append([0] * pad + [1] * len(w) if pad_left else [1] * len(w) + [0] * pad)
    return ids, mask, sample


def pair_spans(ca, cb, m, stride, strategy, left, overflow):
    """the windows of a sentence pair with contents of ca and cb ids (template ids excluded), HF tokenizers'
    truncate_encodings + Encoding::truncate + Encoding::merge_with: m = max_length - the pair template's ids (None: no
    truncation), strategy 'longest_first' / 'only_first' / 'only_second'.
    -> [((startA, stopA), (startB, stopB))] in HF's order.  Raises ValueError where HF misbehaves or raises."""
    if m is None or ca + cb <= m:
        return [((0, ca), (0, cb))]
    if m <= 0:
        raise ValueError('max_length must exceed the ids of the pair template')
    if strategy == 'longest_first':
        n1, n2 = min(ca, cb), max(ca, cb)
        n2 = n1 if n1 > m else max(n1, m - n1)
        if n1 + n2 > m:
            n1 = m // 2
            n2 = n1 + m % 2
        na, nb = (n2, n1) if ca > cb else (n1, n2)
        na, nb = min(na, ca), min(nb, cb)
    elif strategy in ('only_first', 'only_second'):
        rem = ca + cb - m
        first = strategy == 'only_first'
        if (ca if first else cb) <= rem:
            raise ValueError('sequence to truncate too short to respect the provided max_length')
        na, nb = (ca - rem, cb) if first else (ca, cb - rem)
    else:
        raise ValueError('unknown truncation strategy %r' % (strategy,))
    for n, c in ((na, ca), (nb, cb)):
        if n < c and n == 0:
            raise ValueError('longest_first would cut a sequence to 0 ids')
        if n < c and stride >= n:
            raise ValueError('stride is not smaller than the length a sequence is cut to')
    wa = window_spans(ca, na, stride, left, overflow)
    wb = window_spans(cb, nb, stride, left, overflow)
    if len(wa) * len(wb) > 2 ** 31 - 1:
        raise ValueError('more than 2^31 - 1 windows')
    return ([(wa[0], wb[0])] + [(wa[i], wb[j]) for i in range(1, len(wa)) for j in range(len(wb))] +
            [(wa[0], wb[j]) for j in range(1, len(wb))])


def pair_windows(rows_a, rows_b, bos, eos, pre, mid, post, max_length, stride, strategy, left, overflow, padding, multiple,
                 pad_left, pad_id, truncate=True):
    """rows_a, rows_b: encoder output rows (with their single-template ids bos / eos, or None), row i of each side a pair;
    pre / mid / post: the ids of the pair template `pre $A mid $B post`.
    -> (input_ids [N][L], attention_mask [N][L], overflow_to_sample_mapping [N]) as lists, as windows() returns them"""
    head, tail = (0 if bos is None else 1), (0 if eos is None else 1)
    if len(rows_a) != len(rows_b):
        raise ValueError('both sides must hold the same number of rows')
    m = max_length - len(pre) - len(mid) - len(post) if truncate else None
    if m is not None and m <= 0:
        raise ValueError('max_length must exceed the ids of the pair template')
    if truncate and stride > max_length - head - tail:        # enable_truncation checks the single template's ids
        raise ValueError('stride must not exceed max_length - the single template ids')
    out, sample = [], []
    for r, (ra, rb) in enumerate(zip(rows_a, rows_b)):
        a, b = list(ra)[head:len(ra) - tail], list(rb)[head:len(rb) - tail]
        for (a0, a1), (b0, b1) in pair_spans(len(a), len(b), m, stride, strategy, left, overflow):
            out.append(list(pre) + a[a0:a1] + list(mid) + b[b0:b1] + list(post))
            sample.append(r)
    width = max_length if padding == 'max_length' else max((len(w) for w in out), default=0)
    if multiple:
        width = (width + multiple - 1) // multiple * multiple
    if any(len(w) > width for w in out):
        raise ValueError('a pair is longer than the padded width')
    ids, mask = [], []
    for w in out:
        pad = width - len(w)
        ids.append([pad_id] * pad + w if pad_left else w + [pad_id] * pad)
        mask.append([0] * pad + [1] * len(w) if pad_left else [1] * len(w) + [0] * pad)
    return ids, mask, sample
