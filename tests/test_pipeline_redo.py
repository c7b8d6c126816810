"""The pipelined host paths (Engine.encode_host_pipelined, Engine.pipeline_host_pipelined) at their default chunk sizes
with status-raising rows planted in the first, a middle and the last chunk: every planted chunk is redone through the
plain path while later chunks are in flight, and the whole output equals one plain call over the same rows."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import akshar_oracle as O
import synth_corpus as sc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODELS = os.path.join(ROOT, 'tests', 'golden', 'models')
BPE, SPM = os.path.join(MODELS, 'bpe24k.json'), os.path.join(MODELS, 'spm24k.model')
CHUNK = {0: 64 << 20, 1: 128 << 20}          # the defaults of encode_host_pipelined (BPE, Unigram)
PIPE_CHUNK = 64 << 20                        # the default of pipeline_host_pipelined
# rows that make a chunk's fast call raise a status bit:
#   a row start and a word start at every byte, and single-byte words: more events than a warp tile's slots (overflow)
#   3000 alternating vowel signs after one consonant: one grapheme cluster longer than the segmenters' look-back
#   limit, which normalize_text keeps (no code point three times in a row)
PLANTED = ['a'] * 2000 + ['a.b,c!d' * 300, 'a b c d ' * 400, 'क' + 'ु' * 3000,
                          'क' + 'ुू' * 1500 + 'ख']


def _np(t):
    return t.cpu().numpy()


@pytest.fixture(scope='module')
def A():
    import torch
    assert torch.cuda.is_available(), 'GPU tests need a CUDA device'
    import __graft_entry__ as g
    g.build()
    import akshar_b200
    return akshar_b200


@pytest.fixture(scope='module')
def social():
    return sc.Corpus('social', 91).generate(320 << 20)


def plant(data, off, chunk_bytes):
    """PLANTED rows in the middle of the first, a middle and the last chunk of rows cut at chunk_bytes ->
    (pinned data, pinned offsets, indices of the planted chunks, the planted rows' first indices)"""
    import torch
    from akshar_b200 import shard
    ranges = shard.chunk_rows(off, chunk_bytes)
    ks = sorted({0, len(ranges) // 2, len(ranges) - 1})
    at = [(ranges[k][0] + ranges[k][1]) // 2 for k in ks]
    d_p, o_p = sc.pack(PLANTED)
    parts, offs, prev, shift, firsts = [], [off[:1]], 0, 0, []
    for r in at:
        parts += [data[off[prev]:off[r]], d_p]
        offs += [off[prev + 1:r + 1] + shift, o_p[1:] + off[r] + shift]
        firsts.append(r + len(firsts) * len(PLANTED))
        shift += int(o_p[-1])
        prev = r
    parts.append(data[off[prev]:])
    offs.append(off[prev + 1:] + shift)
    d2, o2 = np.concatenate(parts), np.concatenate(offs)
    new = shard.chunk_rows(o2, chunk_bytes)
    assert len(new) == len(ranges) >= 3
    for k, r in zip(ks, firsts):
        assert new[k][0] <= r and r + len(PLANTED) <= new[k][1]
        assert np.array_equal(d2[o2[r]:o2[r + len(PLANTED)]], d_p)
    return torch.from_numpy(d2).pin_memory(), torch.from_numpy(o2).pin_memory(), ks, new, firsts


def sample_rows(ranges, ks, firsts, seed):
    """2000 seeded rows of the planted chunks and the planted rows (not the 9 kB cluster: the oracle is slow on it)"""
    rng = np.random.default_rng(seed)
    rows = np.concatenate([np.arange(*ranges[k]) for k in ks])
    pick = set(rng.choice(rows, size=2000, replace=False).tolist())
    for r in firsts:
        pick.update(range(r + 1995, r + len(PLANTED) - 1))
    return sorted(pick)


@pytest.mark.parametrize('kind', [0, 1], ids=['bpe', 'unigram'])
def test_encode_redo_equals_one_call(A, social, kind):
    """encode_host_pipelined (wide and, for BPE, compact) == tokenizer_encode_batch over the same rows in one call; each
    planted chunk is redone exactly once"""
    data, off = social
    hd, ho, ks, ranges, firsts = plant(data, off, CHUNK[kind])
    om = O.BpeModel(BPE) if kind == 0 else O.UnigramModel(SPM)
    model_ids = (lambda s: O.bpe_encode(om, s)) if kind == 0 else (lambda s: O.unigram_encode(om, s))
    ref = None
    for compact in ((False, True) if kind == 0 else (False,)):
        # a fresh engine: the workspace an earlier redo grew would give the dense rows enough event slots
        eng = A.Engine(0)
        (eng.load_bpe if kind == 0 else eng.load_spm)(BPE if kind == 0 else SPM)
        out = eng.encode_host_pipelined(hd, ho, kind, chunk_bytes=CHUNK[kind], compact=compact)
        assert getattr(eng, 'redone_chunks', 0) == len(ks)
        if compact:
            ids, splits = out.ids().astype(np.int32), out.row_splits()
        else:
            ids, splits = out[0].numpy().copy(), out[1].numpy().copy()
        if ref is None:
            r, _ = eng.tokenizer_encode_batch((hd, ho), kind)
            ref = _np(r.values), _np(r.splits)
        assert np.array_equal(splits, ref[1]) and np.array_equal(ids, ref[0]), 'compact=%s' % compact
    b = hd.numpy().tobytes()
    o = ho.numpy()
    for i in sample_rows(ranges, ks, firsts, 5 + kind):
        e = O.normalize_text(b[o[i]:o[i + 1]].decode('utf-8'))
        assert ref[0][ref[1][i]:ref[1][i + 1]].tolist() == model_ids(e), i


def test_pipeline_redo_equals_two_calls(A, social):
    """pipeline_host_pipelined (normalized text, offsets, cluster and run ends and tags) == normalize_batch +
    segment_batch over the same rows; each planted chunk is redone exactly once"""
    data, off = social
    hd, ho, ks, ranges, firsts = plant(data, off, PIPE_CHUNK)
    eng = A.Engine(0)
    out = eng.pipeline_host_pipelined(hd, ho, chunk_bytes=PIPE_CHUNK)
    assert getattr(eng, 'redone_chunks', 0) == len(ks)
    norm = eng.normalize_batch((hd, ho))
    cl, ru = eng.segment_batch(norm, clusters=True, runs=True)
    nb, no = _np(norm.data[:norm.end]), _np(norm.offsets)
    assert out.norm.numel() == norm.end and np.array_equal(out.norm.numpy(), nb)
    assert np.array_equal(out.offsets.numpy(), no)
    ce, cs = out.cluster_ends()
    assert np.array_equal(cs, _np(cl.splits)) and np.array_equal(ce, _np(cl.values))
    re_, rs, rt = out.run_ends()
    assert np.array_equal(rs, _np(ru.splits)) and np.array_equal(re_, _np(ru.values)) and np.array_equal(rt, _np(ru.extra))
    b, nbb = hd.numpy().tobytes(), nb.tobytes()
    o = ho.numpy()
    for i in sample_rows(ranges, ks, firsts, 7):
        e = O.normalize_text(b[o[i]:o[i + 1]].decode('utf-8'))
        assert nbb[no[i]:no[i + 1]].decode('utf-8') == e, i
        cps = [ord(c) for c in e]
        assert ce[cs[i]:cs[i + 1]].tolist() == O.cp_ends_to_byte_ends(cps, O.segment_breaks(cps)), i


@pytest.mark.parametrize('kind', [0, 1], ids=['bpe', 'unigram'])
def test_slot_overflow_reports_no_stale_id_total(A, kind):
    """a warp tile that runs out of event slots stops the model stage of tokenizer_encode_batch: the id total it reports
    is then 0, not a sum over per-warp-tile counts the stage never wrote (the engine sizes its retry by that total);
    the retry gives the oracle's ids"""
    import torch
    eng = A.Engine(0)
    (eng.load_bpe if kind == 0 else eng.load_spm)(BPE if kind == 0 else SPM)
    lines = sc.Corpus('social', 92).lines(4 << 20) + ['a'] * 2000 + ['a.b,c!d' * 300, 'a b c d ' * 400, 'kya haal hai']
    data, off = sc.pack(lines)
    n = int(off[-1])
    need = eng.lib.akshar_workspace_bytes(n + (n >> 3) + 1024, len(lines))
    eng._ws = torch.full((need + (need >> 3),), 0x7F, dtype=torch.uint8, device=eng.device)   # stale counts everywhere
    ids, _, result = eng.tokenizer_encode_batch((torch.from_numpy(data), torch.from_numpy(off)), kind, check=False)
    r = result.cpu().tolist()
    assert r[2] == A._lib.ST_OVERFLOW and r[3] > 256 and r[0] == 0, r
    ids, _ = eng.tokenizer_encode_batch((torch.from_numpy(data), torch.from_numpy(off)), kind)
    v, sp = _np(ids.values), _np(ids.splits)
    om = O.BpeModel(BPE) if kind == 0 else O.UnigramModel(SPM)
    enc = (lambda s: O.bpe_encode(om, s)) if kind == 0 else (lambda s: O.unigram_encode(om, s))
    for i in list(range(0, len(lines) - 2003, 97)) + list(range(len(lines) - 2003, len(lines))):
        assert v[sp[i]:sp[i + 1]].tolist() == enc(O.normalize_text(lines[i])), i
