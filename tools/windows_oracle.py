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
