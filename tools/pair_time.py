#!/usr/bin/env python
"""Device time of the sentence-pair windows (CUDA events) in the shape of extractive QA on the 1 GiB Hinglish batch of
bench.py: one short row (the question) against every document of 512 rows (the context), only_second, max_length 384,
stride 128.  In one process and in alternated rounds: akshar_pair_windows_write, akshar_windows_write of the contexts
alone with the same max_length and stride, and a fill_ of the pair output's tensors; then what
encode_batch_tensors(texts, text_pair=...) adds to encode_batch(texts + pairs, as_device=True) for 4096 pairs."""
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
    ml, stride = 384, 128
    card = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = 'unknown'
    tk = A.aksharTokenizer(os.path.join(ROOT, 'tests', 'golden', 'models', 'bpe24k.json'), 'bpe')
    eng = tk._eng
    dev = eng.device
    data, off = sc.Corpus('hinglish', 20261018).generate(mb << 20)
    enc, _ = eng.tokenizer_encode_batch((torch.from_numpy(data), torch.from_numpy(off)), 0)
    del data, off
    n_rows = enc.splits.numel() - 1
    docs = torch.cat([enc.splits[::512], enc.splits[-1:]]) if n_rows % 512 else enc.splits[::512]
    n_docs = docs.numel() - 1
    # one question per document: a row of at most 64 content ids, gathered into a ragged side of its own
    lens = enc.splits[1:] - enc.splits[:-1]
    short = torch.nonzero(lens <= 66).flatten()
    q = short[torch.arange(n_docs, device=dev) % short.numel()]
    qlen = lens[q]
    qsplits = torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), torch.cumsum(qlen, 0)])
    qpos = torch.repeat_interleave(enc.splits[q] - qsplits[:-1], qlen) + torch.arange(int(qsplits[-1]), device=dev)
    qvals = enc.values[qpos].contiguous()
    kw = dict(max_length=ml, truncation='only_second', stride=stride, return_overflowing_tokens=True, padding='max_length')
    out = eng.windows_batch((qvals, qsplits), 0, pair_ids=(enc.values, docs), **kw)
    n = out['input_ids'].shape[0]
    skw = dict(max_length=ml, truncation=True, stride=stride, return_overflowing_tokens=True, padding='max_length')
    sout = eng.windows_batch((enc.values, docs), 0, **skw)
    ns = sout['input_ids'].shape[0]

    def splits_of(count, flags, pair):
        wsplits = torch.empty(n_docs + 1, dtype=torch.int64, device=dev)
        result = torch.empty(4, dtype=torch.int64, device=dev)
        ws = torch.empty(eng.lib.akshar_windows_workspace_bytes(n_docs), dtype=torch.uint8, device=dev)
        if pair:
            rc = count(eng._h, 0, qvals.data_ptr(), qsplits.data_ptr(), enc.values.data_ptr(), docs.data_ptr(), 0, n_docs, ml, stride,
                       flags, wsplits.data_ptr(), result.data_ptr(), ws.data_ptr(), ws.numel(), eng._stream())
        else:
            rc = count(eng._h, 0, enc.values.data_ptr(), 0, docs.data_ptr(), n_docs, ml, stride, flags, wsplits.data_ptr(),
                       result.data_ptr(), ws.data_ptr(), ws.numel(), eng._stream())
        assert rc == 0
        return wsplits, int(result[0])
    pflags = C.WIN_TRUNCATE | C.WIN_OVERFLOW | C.WIN_ONLY_SECOND
    sflags = C.WIN_TRUNCATE | C.WIN_OVERFLOW
    pw, pn = splits_of(eng.lib.akshar_pair_windows_count, pflags, True)
    sw, sn = splits_of(eng.lib.akshar_windows_count, sflags, False)
    assert pn == n and sn == ns
    ids, mask, smp = out['input_ids'], out['attention_mask'], out['overflow_to_sample_mapping']
    sids, smask, ssmp = sout['input_ids'], sout['attention_mask'], sout['overflow_to_sample_mapping']

    def pair_write():
        rc = eng.lib.akshar_pair_windows_write(eng._h, 0, qvals.data_ptr(), qsplits.data_ptr(), enc.values.data_ptr(), docs.data_ptr(), 0,
                                               pw.data_ptr(), n_docs, n, ml, stride, pflags, ml, 0, ids.data_ptr(), mask.data_ptr(),
                                               smp.data_ptr(), eng._stream())
        assert rc == 0

    def single_write():
        rc = eng.lib.akshar_windows_write(eng._h, 0, enc.values.data_ptr(), 0, docs.data_ptr(), sw.data_ptr(), n_docs, ns, ml, stride,
                                          sflags, ml, 0, sids.data_ptr(), smask.data_ptr(), ssmp.data_ptr(), eng._stream())
        assert rc == 0

    def fill():
        ids.fill_(0)
        mask.fill_(1)
        smp.fill_(0)
    rounds = [(timed(pair_write), timed(single_write), timed(fill)) for _ in range(5)]
    t_pair = sorted(r[0] for r in rounds)[2]
    t_single = sorted(r[1] for r in rounds)[2]
    t_fill = sorted(r[2] for r in rounds)[2]
    gb, sgb = (2 * n * ml + n) * 8 / 1e9, (2 * ns * ml + ns) * 8 / 1e9
    print('card: %s, power limit %s' % (card, power))
    print('batch: %d rows, %d ids, %d documents; pairs (question, document), only_second, max_length %d, stride %d' %
          (n_rows, enc.values.numel(), n_docs, ml, stride))
    print('akshar_pair_windows_write  %d windows, %.2f GB  %.3f ms  (%.0f GB/s written)' % (n, gb, t_pair, gb / t_pair * 1e3))
    print('akshar_windows_write       %d windows, %.2f GB  %.3f ms  (%.0f GB/s written)' % (ns, sgb, t_single, sgb / t_single * 1e3))
    print('fill_ of the pair output   %.3f ms  (%.0f GB/s written)' % (t_fill, gb / t_fill * 1e3))
    print('pair / single per output byte %.3fx; pair / fill %.2fx (medians of 5 alternated rounds of 10 calls)' %
          ((t_pair / gb) / (t_single / sgb), t_pair / t_fill))
    # what encode_batch_tensors with pairs adds to encoding the texts and pairs in one call
    lines = sc.Corpus('hinglish', 20261018).lines(4 << 20)
    texts, pairs = lines[:4096], lines[4096:8192]

    def host_ms(fn, reps=20):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / reps * 1e3
    wkw = dict(max_length=512, truncation=True, padding='longest')
    enc_only = lambda: tk.encode_batch(texts + pairs, as_device=True)          # noqa: E731
    tensors = lambda: tk.encode_batch_tensors(texts, text_pair=pairs, **wkw)   # noqa: E731
    enc_only(), tensors()
    rounds = [(host_ms(enc_only), host_ms(tensors)) for _ in range(15)]          # alternated: the host is shared
    t_enc = sorted(a for a, _ in rounds)[7]
    t_ten = sorted(b for _, b in rounds)[7]
    d = sorted(b - a for a, b in rounds)
    print('4096 pairs: encode_batch(texts + pairs, as_device=True) %.3f ms, encode_batch_tensors(texts, text_pair, truncation 512, '
          'longest) %.3f ms (medians of 15 alternated rounds of 20 calls); added: median %.3f ms, spread %.3f .. %.3f ms' %
          (t_enc, t_ten, d[7], d[0], d[-1]))


if __name__ == '__main__':
    main()
