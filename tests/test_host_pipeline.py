"""Branches of the pipelined host paths (Engine.encode_host_pipelined, Engine.pipeline_host_pipelined) that the parity and
redo tests do not reach: caller-supplied result buffers, the engine-owned ids buffer growing during a call, and one
engine alternating between the paths."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import synth_corpus as sc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BPE = os.path.join(ROOT, 'tests', 'golden', 'models', 'bpe24k.json')
CHUNK = 1 << 20
DENSE = 'a.b,c!d' * 4          # about one id per byte: more than the half a byte (+ 2 per row) the ids buffer starts with


@pytest.fixture(scope='module')
def A():
    import torch
    assert torch.cuda.is_available(), 'GPU tests need a CUDA device'
    import __graft_entry__ as g
    g.build()
    import akshar_b200
    return akshar_b200


def bpe_engine(A):
    eng = A.Engine(0)
    eng.load_bpe(BPE)
    return eng


def pinned(lines):
    import torch
    data, off = sc.pack(lines)
    return torch.from_numpy(data).pin_memory(), torch.from_numpy(off).pin_memory()


def one_call(eng, hd, ho):
    r, _ = eng.tokenizer_encode_batch((hd, ho), 0)
    return r.values.cpu().numpy(), r.splits.cpu().numpy()


def test_caller_buffers(A):
    """results land in caller-supplied pinned out_ids / out_splits, wide and compact; a buffer that is too small or of the
    wrong dtype is refused with ValueError, never swapped"""
    import torch
    eng = bpe_engine(A)
    hd, ho = pinned(sc.Corpus('social', 31).lines(3 << 20))
    ref_ids, ref_sp = one_call(eng, hd, ho)
    n_rows, n_ids = ho.numel() - 1, ref_ids.size
    for compact, id_dt, sp_dt in ((False, torch.int32, torch.int64), (True, torch.int16, torch.int32)):
        oi = torch.full((n_ids + 100,), -1, dtype=id_dt).pin_memory()
        osp = torch.full((n_rows + 1,), -1, dtype=sp_dt).pin_memory()
        out = eng.encode_host_pipelined(hd, ho, 0, chunk_bytes=CHUNK, out_ids=oi, out_splits=osp, compact=compact)
        if compact:
            assert out.ids16.data_ptr() == oi.data_ptr() and out.splits32.data_ptr() == osp.data_ptr()
            assert np.array_equal(out.ids().astype(np.int32), ref_ids) and np.array_equal(out.row_splits(), ref_sp)
        else:
            assert out[0].data_ptr() == oi.data_ptr() and out[1].data_ptr() == osp.data_ptr()
            assert np.array_equal(out[0].numpy(), ref_ids) and np.array_equal(out[1].numpy(), ref_sp)
        assert (oi[n_ids:] == -1).all()
        other_id, other_sp = (torch.int32, torch.int64) if compact else (torch.int16, torch.int32)
        bad = [dict(out_ids=torch.empty(n_ids - 1, dtype=id_dt).pin_memory()),
               dict(out_ids=torch.empty(n_ids, dtype=other_id).pin_memory()),
               dict(out_splits=torch.empty(n_rows, dtype=sp_dt).pin_memory()),
               dict(out_splits=torch.empty(n_rows + 1, dtype=other_sp).pin_memory())]
        for kw in bad:
            with pytest.raises(ValueError):
                eng.encode_host_pipelined(hd, ho, 0, chunk_bytes=CHUNK, compact=compact, **kw)
    out = eng.encode_host_pipelined(hd, ho, 0, chunk_bytes=CHUNK)        # the engine is still usable after a refusal
    assert np.array_equal(out[0].numpy(), ref_ids) and np.array_equal(out[1].numpy(), ref_sp)


@pytest.mark.parametrize('where', ['last', 'middle'])
def test_ids_buffer_grows_mid_call(A, where):
    """rows of about one id per byte outgrow the ids buffer the engine sizes for the whole batch; it grows while chunks
    are in flight (in the last chunk, or in a middle chunk with another one after it) and the ids equal one plain call"""
    eng = bpe_engine(A)
    if where == 'last':         # 2 chunks: half normal text and half dense rows, then dense rows only
        hd, ho = pinned(sc.Corpus('social', 32).lines(512 << 10) + [DENSE] * ((3 << 20) // 2 // len(DENSE)))
    else:                       # 3 chunks: dense rows, dense rows (the buffer grows), normal text
        hd, ho = pinned([DENSE] * ((2 << 20) // len(DENSE)) + sc.Corpus('social', 32).lines(1 << 20))
    total, n_rows = int(ho[-1]), ho.numel() - 1
    n_chunks = 2 if where == 'last' else 3
    ids, splits = eng.encode_host_pipelined(hd, ho, 0, chunk_bytes=total // n_chunks + 1)
    ids, splits = ids.numpy().copy(), splits.numpy().copy()
    start = (total >> 1) + 2 * n_rows + 1024                 # the ids a fresh engine's buffer holds for this batch
    assert ids.size > start, 'the ids buffer did not have to grow'
    ref_ids, ref_sp = one_call(eng, hd, ho)
    assert np.array_equal(splits, ref_sp) and np.array_equal(ids, ref_ids)


def test_alternating_paths(A):
    """one engine alternating encode (wide, compact) and normalize -> segment: each call gives what its path gives on an
    engine of its own"""
    data, off = sc.Corpus('social', 33).generate(5 << 20)
    import torch
    hd, ho = torch.from_numpy(data).pin_memory(), torch.from_numpy(off).pin_memory()

    def run(eng, what):
        if what == 'wide':
            i, s = eng.encode_host_pipelined(hd, ho, 0, chunk_bytes=CHUNK)
            return [i.numpy().copy(), s.numpy().copy()]
        if what == 'compact':
            c = eng.encode_host_pipelined(hd, ho, 0, chunk_bytes=CHUNK, compact=True)
            return [c.ids().copy(), c.row_splits()]
        p = eng.pipeline_host_pipelined(hd, ho, chunk_bytes=CHUNK)
        ce, cs = p.cluster_ends()
        re_, rs, rt = p.run_ends()
        return [p.norm.numpy().copy(), p.offsets.numpy().copy(), ce, cs, re_, rs, rt]

    alone = {w: run(bpe_engine(A), w) for w in ('wide', 'compact', 'pipe')}
    eng = bpe_engine(A)
    for w in ('wide', 'pipe', 'compact', 'pipe', 'wide', 'compact', 'wide'):
        got = run(eng, w)
        assert all(np.array_equal(g, a) for g, a in zip(got, alone[w])), w
