#!/usr/bin/env python
"""Device time of the packed language-model batches (CUDA events): akshar_pack_count (count + scan) and
akshar_pack_write over the 1 GiB Hinglish batch of bench.py, int32 and uint16 ids, block sizes 2048 and 8192, every
output on; next to a fill_ of the same output tensors and to the same outputs composed from torch ops in the same
process; then what encode_batch_packed adds to encode_batch(as_device=True) for 4096 rows of that batch."""
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'tools')]
import torch  # noqa: E402

import akshar_b200 as A  # noqa: E402
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


def torch_pack(values, splits, L):
    """the same outputs from torch ops: what a user composes without pack_batch (two synchronisations: the boolean index
    and nonzero)"""
    T = values.numel()
    NL = T // L * L
    ids = values[:NL].to(torch.int64)
    starts = splits[:-1][splits[1:] > splits[:-1]] - splits[0]
    first = torch.zeros(NL, dtype=torch.bool, device=values.device)
    first[::L] = True
    first[starts[starts < NL]] = True
    seq = torch.cumsum(first, 0) - 1
    ps = torch.nonzero(first).flatten()
    pos = torch.arange(NL, device=values.device) - ps[seq]
    labels = torch.where(pos == 0, -100, ids)
    cu = torch.cat([ps, torch.tensor([NL], device=values.device)]).to(torch.int32)
    return ids.view(-1, L), labels.view(-1, L), pos.view(-1, L), seq.to(torch.int32).view(-1, L), cu


def main():
    mb = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
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
    del data, off
    n_rows, T = enc.splits.numel() - 1, enc.values.numel()
    print('card: %s, power limit %s' % (card, power))
    print('batch: %d rows, %d ids (%.2f ids per row)' % (n_rows, T, T / n_rows))
    kw = dict(return_position_ids=True, return_seq_idx=True, return_flash_attn_kwargs=True)
    u16 = enc.values.to(torch.int16)                 # compact ids (every id here is below 2^15)
    for L in (2048, 8192):
        for name, vals in (('int32', enc.values), ('uint16', u16)):
            batch, rest = eng.pack_batch((vals, enc.splits), L, **kw)
            n, P = batch['input_ids'].shape[0], batch['cu_seq_lens_q'].numel() - 1
            F = rest.splits.numel() - 1
            ws = eng._ws
            result = torch.empty(8, dtype=torch.int64, device=eng.device)
            flag = 0 if vals.dtype == torch.int32 else 1
            args = (vals.data_ptr(), flag, enc.splits.data_ptr(), n_rows, None, None, 0, L, -1)

            def count():
                assert eng.lib.akshar_pack_count(eng._h, *args, result.data_ptr(), ws.data_ptr(), ws.numel(), eng._stream()) == 0
            outs = [batch[k] for k in ('input_ids', 'labels', 'position_ids', 'seq_idx', 'cu_seq_lens_q')] + [rest.values, rest.splits]

            def write():
                assert eng.lib.akshar_pack_write(eng._h, *args, -100, T, P, F, *[t.data_ptr() for t in outs[:5]],
                                                 rest.values.data_ptr() if rest.values.numel() else None, rest.splits.data_ptr(),
                                                 ws.data_ptr(), ws.numel(), eng._stream()) == 0

            def fill():
                for t in outs:
                    t.fill_(1)
            t_count, t_write, t_fill = timed(count), timed(write), timed(fill)
            gb = sum(t.numel() * t.element_size() for t in outs) / 1e9
            line = ('L=%d %s: %d blocks, %d pieces, output %.2f GB (%.1f B per id); count + scan %.3f ms, write %.3f ms '
                    '(%.0f GB/s), fill_ %.3f ms (%.0f GB/s), write / fill %.2fx' %
                    (L, name, n, P, gb, gb * 1e9 / T, t_count, t_write, gb / t_write * 1e3, t_fill, gb / t_fill * 1e3, t_write / t_fill))
            if name == 'int32':
                write()                                     # the fill_ above overwrote the outputs
                want = torch_pack(enc.values, enc.splits, L)
                for a, b in zip(want, outs[:5]):
                    assert torch.equal(a.view(-1), b.view(-1))
                t_torch = timed(lambda: torch_pack(enc.values, enc.splits, L), reps=3)
                line += '; torch ops %.3f ms (%.1fx the write)' % (t_torch, t_torch / t_write)
            print(line)
            del batch, rest, outs
    # what encode_batch_packed adds to encode_batch(as_device=True): host clock around calls that end in a synchronise
    texts = sc.Corpus('hinglish', 20261018).lines(1 << 20)[:4096]

    def host_ms(fn, reps=20):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / reps * 1e3
    enc_only = lambda: tk.encode_batch(texts, as_device=True)          # noqa: E731
    packed = lambda: tk.encode_batch_packed(texts, 2048, **kw)          # noqa: E731
    enc_only(), packed()
    rounds = [(host_ms(enc_only), host_ms(packed)) for _ in range(15)]          # alternated: the host is shared
    t_enc = sorted(a for a, _ in rounds)[7]
    t_pk = sorted(b for _, b in rounds)[7]
    d = sorted(b - a for a, b in rounds)
    print('4096 rows: encode_batch(as_device=True) %.3f ms, encode_batch_packed (L 2048, every output) %.3f ms (medians of '
          '15 alternated rounds of 20 calls); added: median %.3f ms, spread %.3f .. %.3f ms' % (t_enc, t_pk, d[7], d[0], d[-1]))


if __name__ == '__main__':
    main()
