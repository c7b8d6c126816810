#!/usr/bin/env python
"""Device time of the model-ready windows (CUDA events): akshar_windows_write over the 1 GiB Hinglish batch of bench.py
grouped into long documents (every 512th row split: each document still begins with <s> and ends with </s>), next to a
fill_ of output tensors of the same size in the same process; then what encode_batch_tensors adds to
encode_batch(as_device=True) for 4096 rows of that batch."""
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'tools')]
import torch  # noqa: E402

import akshar_b200 as A  # noqa: E402
from akshar_b200 import _lib as C  # noqa: E402
import synth_corpus as sc  # noqa: E402


def timed(fn, reps=10):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    mb = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
    ml, stride = 512, 128
    card = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = 'unknown'
    tk = A.aksharTokenizer(os.path.join(ROOT, 'tests', 'golden', 'models', 'bpe24k.json'), 'bpe')
    eng = tk._eng
    data, off = sc.Corpus('hinglish', 20261018).generate(mb << 20)
    enc, _ = eng.tokenizer_encode_batch((torch.from_numpy(data), torch.from_numpy(off)), 0)
    n_rows = enc.splits.numel() - 1
    docs = torch.cat([enc.splits[::512], enc.splits[-1:]]) if n_rows % 512 else enc.splits[::512]
    n_docs = docs.numel() - 1
    kw = dict(max_length=ml, truncation=True, stride=stride, return_overflowing_tokens=True, padding='max_length')
    out = eng.windows_batch((enc.values, docs), 0, **kw)
    n = out['input_ids'].shape[0]
    # the window splits of the documents, for calling the write kernel alone
    wsplits = torch.empty(n_docs + 1, dtype=torch.int64, device=eng.device)
    result = torch.empty(4, dtype=torch.int64, device=eng.device)
    ws = torch.empty(eng.lib.akshar_windows_workspace_bytes(n_docs), dtype=torch.uint8, device=eng.device)
    flags = C.WIN_TRUNCATE | C.WIN_OVERFLOW
    rc = eng.lib.akshar_windows_count(eng._h, 0, enc.values.data_ptr(), 0, docs.data_ptr(), n_docs, ml, stride, flags,
                                      wsplits.data_ptr(), result.data_ptr(), ws.data_ptr(), ws.numel(), eng._stream())
    assert rc == 0 and int(result[0]) == n
    ids, mask, smp = out['input_ids'], out['attention_mask'], out['overflow_to_sample_mapping']

    def write():
        rc = eng.lib.akshar_windows_write(eng._h, 0, enc.values.data_ptr(), 0, docs.data_ptr(), wsplits.data_ptr(), n_docs, n, ml,
                                          stride, flags, ml, 0, ids.data_ptr(), mask.data_ptr(), smp.data_ptr(), eng._stream())
        assert rc == 0

    def fill():
        ids.fill_(0)
        mask.fill_(1)
        smp.fill_(0)
    t_write, t_fill = timed(write), timed(fill)
    assert torch.equal(eng.windows_batch((enc.values, docs), 0, **kw)['input_ids'][:, 0], torch.full((n,), 2, device=eng.device))
    gb = (2 * n * ml + n) * 8 / 1e9
    print('card: %s, power limit %s' % (card, power))
    print('batch: %d rows, %d ids, %d documents -> %d windows of %d (stride %d), output %.2f GB' %
          (n_rows, enc.values.numel(), n_docs, n, ml, stride, gb))
    print('akshar_windows_write  %.3f ms  (%.0f GB/s written)' % (t_write, gb / t_write * 1e3))
    print('fill_ of the same     %.3f ms  (%.0f GB/s written)' % (t_fill, gb / t_fill * 1e3))
    print('write / fill          %.2fx' % (t_write / t_fill))
    # what encode_batch_tensors adds to encode_batch(as_device=True): host clock around calls that end in a synchronise
    texts = sc.Corpus('hinglish', 20261018).lines(1 << 20)[:4096]

    def host_ms(fn, reps=20):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / reps * 1e3
    wkw = dict(max_length=ml, truncation=True, padding='longest')
    enc_only = lambda: tk.encode_batch(texts, as_device=True)          # noqa: E731
    tensors = lambda: tk.encode_batch_tensors(texts, **wkw)            # noqa: E731
    enc_only(), tensors()
    rounds = [(host_ms(enc_only), host_ms(tensors)) for _ in range(15)]          # alternated: the host is shared
    t_enc = sorted(a for a, _ in rounds)[7]
    t_ten = sorted(b for _, b in rounds)[7]
    d = sorted(b - a for a, b in rounds)
    print('4096 rows: encode_batch(as_device=True) %.3f ms, encode_batch_tensors (truncation 512, longest) %.3f ms (medians of '
          '15 alternated rounds of 20 calls); added: median %.3f ms, spread %.3f .. %.3f ms' % (t_enc, t_ten, d[7], d[0], d[-1]))


if __name__ == '__main__':
    main()
