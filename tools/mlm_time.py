#!/usr/bin/env python
"""Device time of the masked language-model batches (CUDA events): akshar_mlm_mask over the 1 GiB Hinglish batch of
bench.py as windows 512 / stride 128 (of 512-row documents, as tools/window_time.py cuts them) and as packed blocks of
2048, at the default probabilities; next to a labels.copy_(input_ids) of the same tensors and to the same masking composed from torch ops on the device; transformers'
collator on CPU tensors for 4096 rows; then what encode_batch_mlm adds to encode_batch(as_device=True) for 4096 rows."""
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'tools')]
import torch  # noqa: E402

import akshar_b200 as A  # noqa: E402
from akshar_b200.batch import mlm_thresholds  # noqa: E402
import synth_corpus as sc  # noqa: E402

BPE = os.path.join(ROOT, 'tests', 'golden', 'models', 'bpe24k.json')


def timed(fn, reps=20):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def torch_mask(ids, specials, mask_id, V, p=.15, m=.8, r=.1):
    """the collator's torch_mask_tokens on device tensors: what a user composes without mlm_mask"""
    special = torch.isin(ids, specials)
    prob = torch.full(ids.shape, p, device=ids.device).masked_fill_(special, 0.0)
    sel = torch.bernoulli(prob).bool()
    labels = torch.where(sel, ids, -100)
    rep = torch.bernoulli(torch.full(ids.shape, m, device=ids.device)).bool() & sel
    ids[rep] = mask_id
    rnd = torch.bernoulli(torch.full(ids.shape, r / (1 - m), device=ids.device)).bool() & sel & ~rep
    words = torch.randint(V, ids.shape, device=ids.device)
    ids[rnd] = words[rnd]
    return ids, labels


def main():
    mb = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
    card = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = 'unknown'
    print('card: %s, power limit %s' % (card, power))
    tk = A.aksharTokenizer(BPE, 'bpe')
    eng = tk._eng
    data, off = sc.Corpus('hinglish', 20261018).generate(mb << 20)
    enc, _ = eng.tokenizer_encode_batch((torch.from_numpy(data), torch.from_numpy(off)), 0)
    del data, off
    print('batch: %d rows, %d ids' % (enc.splits.numel() - 1, enc.values.numel()))
    t = (__import__('ctypes').c_uint64 * 3)(*mlm_thresholds(.15, .8, .1))
    specials = torch.tensor([0, 1, 2, 3, 4], device=eng.device)
    # the windows of section 4.8: the rows grouped into documents of 512 rows (each still begins with <s> and ends with </s>)
    n_rows = enc.splits.numel() - 1
    docs = torch.cat([enc.splits[::512], enc.splits[-1:]]) if n_rows % 512 else enc.splits[::512]
    shapes = (('windows 512 / stride 128', lambda: eng.windows_batch((enc.values, docs), 0, max_length=512, truncation=True,
                                                                       stride=128, return_overflowing_tokens=True)['input_ids']),
              ('packed L = 2048', lambda: eng.pack_batch(enc, 2048)[0]['input_ids']))
    for name, make in shapes:
        ids = make()
        N, L = ids.shape
        labels = torch.empty_like(ids)

        def kernel():
            assert eng.lib.akshar_mlm_mask(eng._h, 0, ids.data_ptr(), N, L, 1234, 0, 0, t, 4, 0, labels.data_ptr(),
                                           eng._stream()) == 0
        t_k = timed(kernel)
        t_c = timed(lambda: labels.copy_(ids))
        t_t = timed(lambda: torch_mask(ids, specials, 4, 24000), reps=3)
        gb = 16 * ids.numel() / 1e9
        print('%s: [%d, %d] = %d positions; mlm kernel %.3f ms (%.0f GB/s of 16 B per position), labels.copy_(input_ids) '
              '%.3f ms (%.0f GB/s), kernel / copy %.2fx; torch ops %.3f ms (%.1fx the kernel)' %
              (name, N, L, ids.numel(), t_k, gb / t_k * 1e3, t_c, gb / t_c * 1e3, t_k / t_c, t_t, t_t / t_k))
        cpu = ids[:4096].cpu()
        del ids, labels
        try:
            from transformers import DataCollatorForLanguageModeling, PreTrainedTokenizerFast
            htok = PreTrainedTokenizerFast(tokenizer_file=BPE, pad_token='<pad>', unk_token='<unk>', bos_token='<s>', eos_token='</s>',
                                           mask_token='<mask>')
            coll = DataCollatorForLanguageModeling(tokenizer=htok, mlm=True)
            coll.torch_mask_tokens(cpu.clone())
            t0 = time.perf_counter()
            for _ in range(5):
                coll.torch_mask_tokens(cpu.clone())
            print('  transformers collator on CPU tensors, %d rows x %d: %.3f ms' % (cpu.shape[0], cpu.shape[1],
                                                                                     (time.perf_counter() - t0) / 5 * 1e3))
        except ImportError:
            print('  transformers collator: not measured (transformers is not installed)')
    # what encode_batch_mlm adds to encode_batch(as_device=True): host clock around calls that end in a synchronise
    texts = sc.Corpus('hinglish', 20261018).lines(1 << 20)[:4096]
    kw = dict(truncation=True, max_length=512, stride=128, return_overflowing_tokens=True)

    def host_ms(fn, reps=20):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / reps * 1e3
    enc_only = lambda: tk.encode_batch(texts, as_device=True)                    # noqa: E731
    tensors = lambda: tk.encode_batch_tensors(texts, **kw)                       # noqa: E731
    masked = lambda: tk.encode_batch_mlm(texts, 1234, **kw)                      # noqa: E731
    enc_only(), tensors(), masked()
    rounds = [(host_ms(enc_only), host_ms(tensors), host_ms(masked)) for _ in range(15)]     # alternated: the host is shared
    med = lambda xs: sorted(xs)[7]                                              # noqa: E731
    d = sorted(c - a for a, _, c in rounds)
    print('4096 rows: encode_batch(as_device=True) %.3f ms, encode_batch_tensors %.3f ms, encode_batch_mlm %.3f ms (medians '
          'of 15 alternated rounds of 20 calls); added over encode_batch: median %.3f ms, spread %.3f .. %.3f ms; over '
          'encode_batch_tensors: median %.3f ms' % (med([a for a, _, _ in rounds]), med([b for _, b, _ in rounds]),
                                                    med([c for _, _, c in rounds]), d[7], d[0], d[-1],
                                                    med([c - b for _, b, c in rounds])))


if __name__ == '__main__':
    main()
