#!/usr/bin/env python
"""bench.py -- the hot path's headline metric on B200 (BASELINE.json): UTF-8 input GB/s (+ tokens/s) of batch encode.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--mb MB] [--workload bpe|unigram|pipeline|mixed]
                  [--dump-outputs DIR]

One step = one pass of aksharTokenizer.encode over one batch: normalize_text -> BPE-24k ids for every row of the
batch (BASELINE.json configs[1]: "BPE vocab 24k batch encode of 1 GB synthetic Hinglish, 1 B200").  Run without
--workload on one GPU, the line also carries `also`: configs[2] (Unigram-24k, 1 GiB Hindi) and configs[3] (normalize +
akshars + script runs, 4 GiB social Hinglish) measured the same way.  With N > 1 every rank (one process per GPU, launched
by torchrun) encodes its own shard of configs[4]'s mixed corpus (2 : 1 : 1 Hinglish / Hindi / social, 4 GiB per GPU = 32 GiB
at N = 8, fed as 1 GiB batches) -- weak scaling, no collective on the data path; only the timing is reduced (max over
ranks).

Prints ONE JSON line.  `value` is device-timed with the input already in HBM; `e2e` is the same metric through the public
batch API from pinned host buffers with the H2D copy of the text and the D2H read of the ids inside the timed region.
`roofline` is the dominant kernel's algorithmic bytes / its CUDA-event time against MEASURED_PEAKS.json (and, per stage,
SURVEY section 8d's bytes over the stage's kernels); `cpu_baseline` is the oracle port of the same path on the host cores
(bounded sample) -- the same rows are compared id for id with the GPU's before anything is timed (`parity_in_run`).
--impl reference times that CPU implementation alone, with every host core.

--dump-outputs DIR writes, after the timed steps, what the last timed step returned as DIR/<workload>_<array>.npy (float32
or float64, 64 MiB at most in all): for a fixed, seeded sample of rows their ids / normalized bytes / mask bits and
their offsets into the full outputs, plus every batch's result counters.  The inputs depend only on the arguments, so two
builds can be compared output for output.  Nothing is written into the source tree (not even bytecode): it may be
read-only, and the library is the one __graft_entry__.build() left there.
"""
import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time
import zlib

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, 'tools')):
    if p not in sys.path:
        sys.path.insert(0, p)

MODELS = os.path.join(ROOT, 'tests', 'golden', 'models')
CHUNK = 32 << 20
SEED = 20261018
KIND = {'bpe': 'hinglish', 'unigram': 'hindi', 'pipeline': 'social', 'mixed': 'mixed'}
MIX = ('hinglish', 'hinglish', 'hindi', 'social')        # configs[4]: 2 : 1 : 1, chunk by chunk


# ------------------------------------------------------------------ synthetic corpus (SURVEY.md section 8d)
_corpus = {}


def _gen_chunk(args):
    kind, index, nbytes = args
    import synth_corpus as sc
    if kind == 'mixed':
        kind = MIX[index % len(MIX)]
    if kind not in _corpus:
        _corpus[kind] = sc.Corpus(kind, SEED)
    return _corpus[kind].chunk(index, nbytes)


def make_corpus(kind, nbytes, first_chunk=0, procs=None):
    """-> (uint8 numpy array, int64 row offsets); chunk indices first_chunk.. (rank-disjoint for the sharded runs)"""
    import numpy as np
    n = max(1, (nbytes + CHUNK - 1) // CHUNK)
    jobs = [(kind, first_chunk + i, min(CHUNK, nbytes - i * CHUNK)) for i in range(n)]
    procs = procs or min(len(jobs), os.cpu_count() or 1)
    if procs > 1:
        with mp.get_context('fork').Pool(procs) as pool:
            parts = pool.map(_gen_chunk, jobs)
    else:
        parts = [_gen_chunk(j) for j in jobs]
    datas, offs, base = [], [np.zeros(1, dtype=np.int64)], 0
    for d, o in parts:
        datas.append(d)
        offs.append(o[1:] + base)
        base += d.size
    return np.concatenate(datas), np.concatenate(offs)


# ------------------------------------------------------------------ CPU arm: the oracle port on the host cores
def _crc(a):
    import numpy as np
    return zlib.crc32(np.ascontiguousarray(a).tobytes())


def _cpu_init(workload):
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import akshar_oracle as O
    global _O, _M
    _O = O
    if workload in ('bpe', 'mixed'):
        _M = O.BpeModel(os.path.join(MODELS, 'bpe24k.json'))
    elif workload == 'unigram':
        _M = O.UnigramModel(os.path.join(MODELS, 'spm24k.model'))
    else:
        _M = None


def _cpu_work(args):
    """-> (token count, one checksum per row of what the reference returns for it)"""
    import numpy as np
    workload, lines = args
    n = 0
    sums = []
    for s in lines:
        norm = _O.normalize_text(s)
        if workload in ('bpe', 'mixed'):
            ids = _O.bpe_encode(_M, norm)
            n += len(ids)
            sums.append(_crc(np.asarray(ids, dtype=np.int32)))
        elif workload == 'unigram':
            ids = _O.unigram_encode(_M, norm)
            n += len(ids)
            sums.append(_crc(np.asarray(ids, dtype=np.int32)))
        else:
            cps = [ord(c) for c in norm]
            ce = _O.cp_ends_to_byte_ends(cps, _O.segment_breaks(cps))
            runs = _O.detect_code_switches(norm)
            n += len(ce) + len(runs)
            sums.append(zlib.crc32(norm.encode('utf-8')) ^ _crc(np.asarray(ce, dtype=np.int32)) ^
                        zlib.crc32(repr([(len(seg.encode('utf-8')), lab) for seg, lab in runs]).encode()))
    return n, sums


class CpuArm:
    """the oracle restatement of the same path, one process per host core, over a bounded sample of the workload"""

    def __init__(self, workload, data, off, sample_bytes):
        import numpy as np
        self.workload = workload
        hi = int(np.searchsorted(off, sample_bytes, side='right'))
        hi = max(1, min(hi, off.size - 1))
        b = data[:off[hi]].tobytes()
        self.lines = [b[off[i]:off[i + 1]].decode('utf-8') for i in range(hi)]
        self.nbytes = int(off[hi])
        self.cores = os.cpu_count() or 1
        self.pool = mp.get_context('fork').Pool(self.cores, initializer=_cpu_init, initargs=(workload,))
        per = max(1, len(self.lines) // (self.cores * 4))
        self.jobs = [(workload, self.lines[i:i + per]) for i in range(0, len(self.lines), per)]
        self.sums = None

    def step(self):
        t = time.perf_counter()
        res = self.pool.map(_cpu_work, self.jobs)
        dt = time.perf_counter() - t
        self.sums = [c for _, s in res for c in s]
        return dt, sum(n for n, _ in res)

    def native_libs(self):
        """the third-party engines the reference delegates to, alone, with their own native batching (SURVEY 8d's
        "fairer second CPU line"): HF tokenizers encode_batch / SentencePiece encode with num_threads on already
        normalized rows.  -> dict, or why it is not available on this box"""
        try:
            sys.path.insert(0, os.path.join(ROOT, 'oracle'))
            import akshar_oracle as O
            norm = [O.normalize_text(s) for s in self.lines[:20000]]
            nb = sum(len(s.encode('utf-8')) for s in norm)
            if self.workload in ('bpe', 'mixed'):
                from tokenizers import Tokenizer
                tk = Tokenizer.from_file(os.path.join(MODELS, 'bpe24k.json'))
                tk.encode_batch(norm[:1000])
                t = time.perf_counter()
                tk.encode_batch(norm)
                what = 'tokenizers.Tokenizer.encode_batch (Rust, rayon) on normalized rows'
            elif self.workload == 'unigram':
                import sentencepiece as spm
                sp = spm.SentencePieceProcessor()
                sp.Load(os.path.join(MODELS, 'spm24k.model'))
                t = time.perf_counter()
                sp.encode(norm, num_threads=self.cores)
                what = 'sentencepiece encode(num_threads=%d) on normalized rows' % self.cores
            else:
                return None
            dt = time.perf_counter() - t
            return {'value': nb / dt / 1e9, 'unit': 'GB/s', 'what': what, 'sample_mb': nb / 1e6}
        except Exception as e:      # library not on this box
            return {'unavailable': repr(e)[:120]}

    def close(self):
        self.pool.close()
        self.pool.join()


# ------------------------------------------------------------------ clocks
class ClockSampler:
    Q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.rows = []             # (arrival time, line)
        self.proc = None
        self.t_from = 0.0
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits',
                                          '-lms', '20'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def wait_first(self, timeout=5.0):
        """nvidia-smi takes a few hundred ms to deliver its first line: wait for it so that the (short) measured phases
        are covered"""
        t0 = time.perf_counter()
        while self.proc and not self.rows and time.perf_counter() - t0 < timeout:
            time.sleep(0.01)

    def mark(self):
        """only samples that arrive from now on count (the measured phases start here)"""
        self.t_from = time.perf_counter()

    def stop(self):
        if not self.proc:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ts, r in self.rows:
            if ts < self.t_from:
                continue
            f = [x.strip() for x in r.split(',')]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': mx, 'reasons': sorted(reasons), 'samples': len(sm)}


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        return float(json.load(open(p))['hbm_gbs']), 'measured'
    return 6650.0, 'fallback'


def traffic_table():
    """DRAM bytes per input byte of each hot kernel from the committed `ncu --set full` summary (profiles/r02_traffic.json:
    (dram__bytes_read.sum + dram__bytes_write.sum) / input bytes at the size stated there)"""
    p = os.path.join(ROOT, 'profiles', 'r02_traffic.json')
    if os.path.exists(p):
        return json.load(open(p))
    return {}


# ------------------------------------------------------------------ --dump-outputs
DUMP_ROWS = 4096
DUMP_LIMIT = 64 << 20


def dump_rows(n_rows):
    """the rows whose outputs are dumped: a fixed, seeded sample"""
    import numpy as np
    rng = np.random.default_rng(SEED)
    return np.sort(rng.choice(n_rows, size=min(n_rows, DUMP_ROWS), replace=False))


def _spans(lo, hi):
    """flat indices lo[j] .. hi[j] - 1 of every j, concatenated"""
    import numpy as np
    n = hi - lo
    return np.repeat(lo - np.cumsum(n) + n, n) + np.arange(int(n.sum()), dtype=np.int64)


def sample_outputs(outs, ranges, rows, tokens):
    """one step's per-batch outputs ((ids, normalized text, result) or (masks, normalized text, result)), restricted to the
    rows `rows` (global indices) -> {name: float array}"""
    import numpy as np
    import torch
    parts = {}
    for (lo, hi), o in zip(ranges, outs):
        norm = o[1]
        dev = norm.offsets.device
        t = torch.from_numpy(rows[(rows >= lo) & (rows < hi)] - lo).to(dev)
        n0, n1 = norm.offsets[t].cpu().numpy(), norm.offsets[t + 1].cpu().numpy()
        got = {'norm_offsets': np.stack([n0, n1], 1), 'norm': norm.data[torch.from_numpy(_spans(n0, n1)).to(dev)],
               'result': o[-1][None]}
        if tokens:
            s0, s1 = o[0].splits[t].cpu().numpy(), o[0].splits[t + 1].cpu().numpy()
            got['id_splits'] = np.stack([s0, s1], 1)
            got['ids'] = o[0].values[torch.from_numpy(_spans(s0, s1)).to(dev)]
        else:
            # the four mask planes at every byte of a row and at its end (a cluster / run that ends a row sets the bit
            # of the byte after it)
            pos = torch.from_numpy(_spans(n0, n1 + 1)).to(dev)
            planes = (o[0]['cluster'], o[0]['run'], o[0]['tags'][0], o[0]['tags'][1])
            got['masks'] = torch.stack([(p[pos >> 5].to(torch.int64) >> (pos & 31)) & 1 for p in planes])
        for k, v in got.items():
            parts.setdefault(k, []).append(v.cpu().numpy() if torch.is_tensor(v) else v)
    out = {k: np.concatenate(v, axis=-1) if k == 'masks' else np.concatenate(v) for k, v in parts.items()}
    out['rows'] = rows
    wide = ('norm_offsets', 'id_splits', 'result', 'rows')
    return {k: v.astype(np.float64 if k in wide else np.float32) for k, v in out.items()}


def write_dump(path, arrays):
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise RuntimeError('--dump-outputs: %d bytes, more than %d' % (total, DUMP_LIMIT))
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), k
        np.save(os.path.join(path, k + '.npy'), a)


# ------------------------------------------------------------------ one workload on this rank
class Rank:
    def __init__(self):
        self.rank = int(os.environ.get('RANK', '0'))
        self.world = int(os.environ.get('WORLD_SIZE', '1'))
        self.local = int(os.environ.get('LOCAL_RANK', '0'))


def describe(workload, mb, world):
    return {'bpe': 'BPE-24k batch encode (normalize_text -> ids) of %d MiB synthetic Hinglish per GPU' % mb,
            'unigram': 'Unigram-24k Viterbi encode (normalize_text -> ids) of %d MiB synthetic Hindi per GPU' % mb,
            'pipeline': 'normalize + akshars + script runs on %d MiB synthetic social Hinglish per GPU' % mb,
            'mixed': 'sentence-sharded BPE-24k encode of %d MiB per GPU (%d GPUs) of the 2:1:1 Hinglish / Hindi / social mix, '
                     'in 1 GiB batches' % (mb, world)}[workload]


def run_workload(R, workload, mb, steps, warmup, cpu_sample_mb, dist, with_cpu=True, dump=None):
    """-> the JSON line (a dict) on rank 0, None elsewhere; with `dump` (a dict) rank 0 adds the sampled outputs of the last
    timed step to it"""
    import numpy as np
    import torch
    kind = KIND[workload]
    nbytes = mb << 20
    sub = 1 << 30                                   # batches of at most 1 GiB (event positions are 32-bit)
    chunks_per_rank = (nbytes + CHUNK - 1) // CHUNK
    # host-side work that forks (corpus generation, the CPU arm's worker pool) comes first
    data, off = make_corpus(kind, nbytes, R.rank * chunks_per_rank, procs=max(1, (os.cpu_count() or 1) // R.world))
    n_rows = off.size - 1
    arm = CpuArm(workload, data, off, int(cpu_sample_mb * (1 << 20))) if (R.rank == 0 and with_cpu) else None
    import akshar_b200 as A
    from akshar_b200 import shard

    # the rank's shard as batches of <= 1 GiB (row ranges)
    n_sub = max(1, (int(off[-1]) + sub - 1) // sub)
    ranges = [r for r in shard.shard_rows(off, n_sub) if r[1] > r[0]]
    h_batches = []
    for lo, hi in ranges:
        d, o = shard.take_shard(data, off, lo, hi)
        h_batches.append((torch.from_numpy(np.ascontiguousarray(d)).pin_memory(), torch.from_numpy(np.ascontiguousarray(o)).pin_memory()))
    if workload in ('bpe', 'mixed'):
        tk = A.aksharTokenizer(os.path.join(MODELS, 'bpe24k.json'), 'bpe', device=R.local)
        eng, mkind = tk._eng, 0
    elif workload == 'unigram':
        tk = A.aksharTokenizer(os.path.join(MODELS, 'spm24k.model'), 'sentencepiece', device=R.local)
        eng, mkind = tk._eng, 1
    else:
        eng, mkind = A.Engine(R.local), None
    dev_batches = [eng.put(hb) for hb in h_batches]
    torch.cuda.synchronize()

    def device_step(batches):
        outs = []
        for b in batches:
            if mkind is not None:
                outs.append(eng.tokenizer_encode_batch(b, mkind, check=False))
            else:
                # one library call: normalize_text, then akshars + script runs of the normalized rows as bit masks
                # (1 bit per byte and stream + two tag planes); nothing is read back in between
                norm, mk = eng.normalize_segment_batch(b, check=False)
                outs.append((mk, norm, mk['result']))
        return outs

    def offsets_form(b):
        """the same stage through the two-call offset form (int32 ends): what the CPU arm's rows are compared with, and
        what the masks of the timed call must agree with"""
        norm = eng.normalize_batch(b)
        c, r = eng.segment_batch(norm, clusters=True, runs=True)
        return c, r, norm

    def barrier():
        torch.cuda.synchronize()
        if R.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- correctness of the run that is about to be timed: status bits clear, and the CPU arm's rows id for id
    outs = device_step(dev_batches)
    torch.cuda.synchronize()
    n_tokens = n_norm = n_c = n_r = 0
    for o in outs:
        res = o[-1].cpu()
        assert int(res[2]) == 0, 'status bits %d' % int(res[2])
        if mkind is not None:
            n_tokens += int(res[0])
            n_norm += int(res[1])
        else:
            n_c += int(res[0])
            n_r += int(res[1])
            n_norm += int(res[3])
    if mkind is None:
        n_tokens = n_c + n_r
    parity = None
    if arm is not None:
        arm.step()
        k = len(arm.lines)
        o = outs[0]
        if mkind is not None:
            sp = o[0].splits[:k + 1].cpu().numpy()
            iv = o[0].values[:int(sp[-1])].cpu().numpy().astype(np.int32)
            got = [_crc(iv[sp[i]:sp[i + 1]]) for i in range(k)]
        else:
            c, r, norm = offsets_form(dev_batches[0])
            # the timed call's masks == the offset form, bit for bit, over the first 64 MiB of the batch (+ all totals)
            mk = o[0]
            rr = mk['result'].cpu()
            assert int(rr[0]) == c.values.numel() and int(rr[1]) == r.values.numel() and int(rr[3]) == norm.end
            assert torch.equal(o[1].offsets, norm.offsets) and torch.equal(o[1].data[:norm.end], norm.data[:norm.end])
            no_all = norm.offsets.cpu().numpy()
            kk = int(np.searchsorted(no_all, 64 << 20))
            kk = max(1, min(kk, no_all.size - 1))
            lim = int(no_all[kk])
            nw = lim // 32
            for rag, key in ((c, 'cluster'), (r, 'run')):
                sp = rag.splits[:kk + 1].cpu().numpy()
                ev = rag.values[:int(sp[-1])].cpu().numpy().astype(np.int64)
                pos = no_all[np.repeat(np.arange(kk), np.diff(sp))] + ev
                m = np.zeros((lim // 32 + 1) * 32, dtype=bool)
                m[pos] = True
                exp_w = np.packbits(m, bitorder='little').view(np.uint32)[:nw]
                assert np.array_equal(mk[key][:nw].cpu().numpy().view(np.uint32), exp_w), 'mask of the %s ends differs' % key
            del mk
            no = norm.offsets[:k + 1].cpu().numpy()
            nb = norm.data[:int(no[-1])].cpu().numpy()
            cs = c.splits[:k + 1].cpu().numpy()
            ce = c.values[:int(cs[-1])].cpu().numpy().astype(np.int32)
            rs = r.splits[:k + 1].cpu().numpy()
            re_ = r.values[:int(rs[-1])].cpu().numpy()
            rt = r.extra[:int(rs[-1])].cpu().numpy()
            tags = ['devanagari', 'roman', 'digit', 'punct', 'other']
            got = []
            for i in range(k):
                ends = re_[rs[i]:rs[i + 1]].tolist()
                lens = [e - (ends[j - 1] if j else 0) for j, e in enumerate(ends)]
                labs = [None if t == 255 else tags[t] for t in rt[rs[i]:rs[i + 1]].tolist()]
                got.append(zlib.crc32(nb[no[i]:no[i + 1]].tobytes()) ^ _crc(ce[cs[i]:cs[i + 1]]) ^
                           zlib.crc32(repr(list(zip(lens, labs))).encode()))
        bad = [i for i in range(k) if got[i] != arm.sums[i]]
        assert not bad, 'GPU result differs from the CPU reference port on rows %s of the timed batch' % bad[:5]
        parity = k
    del outs
    sampler = ClockSampler(R.local) if R.rank == 0 else None
    if sampler:
        sampler.wait_first()
    for _ in range(max(0, warmup - 1)):
        device_step(dev_batches)
    barrier()
    if sampler:
        sampler.mark()          # clocks are sampled every 20 ms from here to the end of the measured phases (timed steps,
    l0 = eng.launch_count()     # end-to-end steps, per-kernel timing steps)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        last = None             # a step's outputs are freed before the next step allocates, as if they were discarded
        last = device_step(dev_batches)
    e1.record()
    barrier()
    launches = eng.launch_count() - l0
    ms = e0.elapsed_time(e1) / steps
    if dump is not None and R.rank == 0:
        for k, v in sample_outputs(last, ranges, dump_rows(n_rows), mkind is not None).items():
            dump['%s_%s' % (workload, k)] = v
    del last

    # ---- end to end through the public batch API: pinned host text in, ids (or offsets) on the host out
    bufs = {}

    def e2e_step():
        moved = 0
        for hb in h_batches:
            if mkind is not None:
                # the public host -> ids call: H2D of chunk k+1, kernels of chunk k and D2H of chunk k-2 overlap; the ids
                # cross the link as uint16, the row splits as int32 (akshar_tokenizer_encode_batch_ex)
                res = eng.encode_host_pipelined(hb[0], hb[1], mkind, compact=True)
                moved += res.ids16.numel() * 2 + res.splits32.numel() * 4 + 32 * len(res.chunk_ids)
                continue
            # the public host -> host call of this stage: chunks over three streams; back come the normalized text, its row
            # offsets and four mask planes (cluster ends, run ends, two tag planes) of one bit per normalized byte
            po = eng.pipeline_host_pipelined(hb[0], hb[1])
            moved += po.norm.numel() + po.offsets.numel() * 8 + 16 * int(po.chunk_words[-1]) + 32 * (len(po.chunk_rows) - 1)
        return moved

    d2h = e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        d2h = e2e_step()
    barrier()
    e2e_s = (time.perf_counter() - t0) / steps

    # ---- dominant kernel: the library brackets its hot kernels with CUDA events on the launching stream
    # (akshar_timing_enable); average over a few passes over the first batch
    eng.timing(True)
    names = ['ak_nf3_classify_kernel', 'ak_nf_write_kernel'] + (['ak_words_kernel', 'ak_resolve_kernel<bpe>', 'ak_emit_kernel'] if mkind == 0 else
                                                                 ['ak_words_kernel', 'ak_resolve_kernel<unigram>', 'ak_emit_kernel'] if mkind == 1 else
                                                                 ['ak_seg_mask_kernel'])
    acc = {k: [] for k in names}
    for _ in range(3):
        device_step(dev_batches[:1])
        torch.cuda.synchronize()
        for k in names:
            v = eng.kernel_ms(k)
            if v is not None:
                acc[k].append(v)
    eng.timing(False)
    clocks = sampler.stop() if sampler else None
    kms = {k: sum(v) / len(v) for k, v in acc.items() if v}
    # algorithmic bytes per launch (DESIGN.md section 4: what the kernel must read and write once), first batch
    f = dev_batches[0].n_bytes / max(1, int(off[-1]))
    b_in, b_norm, rows1, tok1 = dev_batches[0].n_bytes, n_norm * f, dev_batches[0].n_rows, n_tokens * f
    ev1 = tok1 / 1.25 + rows1                                                   # events: words (1.25 ids each) + row starts
    alg = {
        'ak_nf3_classify_kernel': b_in + 4 * (b_in // 16),                      # text in, one emit mask per 16-byte chunk out
        'ak_nf_write_kernel': b_in + 4 * (b_in // 16) + b_norm + 8 * (rows1 + 1),
        'ak_words_kernel': b_norm + 8 * ev1,                                    # text in, one 8-byte event per word / row out
        'ak_resolve_kernel<bpe>': b_norm + 16 * ev1,                            # the words' bytes + events in, resolved records out
        'ak_resolve_kernel<unigram>': b_norm + 20 * ev1,
        'ak_emit_kernel': 8 * ev1 + 4 * tok1 + 8 * (rows1 + 1),
        'ak_seg_mask_kernel': b_norm + 4 * (b_norm // 8) + 8 * (rows1 + 1),          # text + row offsets in, four planes of 1 bit per byte out
    }
    kern = {k: (kms[k], alg[k]) for k in kms}
    dom = max(kern, key=lambda k: kern[k][0])
    peak, peak_kind = peaks()
    ach = kern[dom][1] / (kern[dom][0] * 1e-3) / 1e9
    # SURVEY 8d's bytes per STAGE over the device time of the whole step: text in + normalized text out + row offsets,
    # and what the stage after it adds (ids, or cluster / run ends)
    if mkind is not None:
        stage_bytes = int(off[-1]) + n_norm + 4 * n_tokens + 2 * 8 * (n_rows + 1)
    else:
        stage_bytes = int(off[-1]) + n_norm + 4 * (n_norm // 8) + 2 * 8 * (n_rows + 1)

    # ---- reduce over ranks
    t = torch.tensor([ms, e2e_s * 1e3], dtype=torch.float64, device='cuda')
    cnt = torch.tensor([int(off[-1]), n_tokens, launches, d2h, int(off[-1]) + 8 * (n_rows + len(h_batches))], dtype=torch.float64, device='cuda')
    if R.world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    ms_max, e2e_ms = float(t[0]), float(t[1])
    tot_bytes, tot_tokens, tot_launch, tot_d2h, tot_h2d = (float(x) for x in cnt)
    if R.rank != 0:
        return None
    cpu = None
    if arm is not None:
        dt, ctok = arm.step()
        cpu = {'value': arm.nbytes / dt / 1e9, 'unit': 'GB/s', 'cores': arm.cores, 'kind': 'port', 'tokens_per_s': ctok / dt,
               'sample': '%d rows / %.1f MB of this workload, oracle/akshar_oracle.py on %d processes, %.1f s'
                         % (len(arm.lines), arm.nbytes / 1e6, arm.cores, dt),
               'native_libs_alone': arm.native_libs()}
        arm.close()
    metric = 'utf8_input_GBps_batch_encode' if workload != 'pipeline' else 'utf8_input_GBps_normalize_segment'
    tt = traffic_table()
    return {
        'metric': metric, 'value': tot_bytes / (ms_max * 1e-3) / 1e9, 'unit': 'GB/s', 'tokens_per_s': tot_tokens / (ms_max * 1e-3),
        'n_gpus': R.world, 'steps': steps, 'warmup': warmup, 'ms_per_step': ms_max, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'u8', 'data': 'synthetic',
        'config': {'workload': describe(workload, mb, R.world), 'bytes_per_gpu': int(off[-1]),
                   'model': {'bpe': 'tests/golden/models/bpe24k.json', 'mixed': 'tests/golden/models/bpe24k.json',
                             'unigram': 'tests/golden/models/spm24k.model', 'pipeline': None}[workload],
                   'l2': 'inputs larger than L2 (no flush needed)' if mb >= 256 else 'input smaller than 2x L2',
                   'sharding': 'sentences, no collective',
                   'word_cache': 'lives as long as the model (as in HF tokenizers); every step still hashes and looks up every word'},
        'rows_per_gpu': n_rows, 'tokens_per_gpu': n_tokens, 'normalized_bytes_per_gpu': n_norm,
        'bytes_per_token': int(off[-1]) / max(1, n_tokens) if mkind is not None else None,
        'parity_in_run': parity is not None, 'rows_compared': parity or 0,
        'e2e': {'value': tot_bytes / (e2e_ms * 1e-3) / 1e9, 'unit': 'GB/s', 'h2d_bytes_per_step': int(tot_h2d / R.world),
                'd2h_bytes_per_step': int(tot_d2h / R.world), 'ms_per_step': e2e_ms, 'chunks_redone': getattr(eng, 'redone_chunks', 0),
                'out': 'uint16 ids + int32 chunk-relative row splits' if mkind is not None else 'normalized text + int64 row offsets + 4 boundary mask planes (1 bit per normalized byte each)'},
        'gpu_launches': int(tot_launch),
        'roofline': {'bound': 'hbm', 'kernel': dom, 'achieved': ach, 'peak': peak, 'peak_source': peak_kind, 'unit': 'GB/s',
                     'frac': ach / peak, 'frac_of_nominal_8000': ach / 8000.0,
                     'traffic': (int(tt[dom]['dram_bytes_per_input_byte'] * b_in) if dom in tt else None),
                     'traffic_source': 'profiles/r02_traffic.json (ncu --set full, dram read + write per input byte, scaled)' if dom in tt else None,
                     'ms': kern[dom][0], 'algorithmic_bytes': kern[dom][1],
                     'kernels_ms': {k: v[0] for k, v in kern.items()},
                     'kernels_frac': {k: v[1] / (v[0] * 1e-3) / 1e9 / peak for k, v in kern.items()},
                     'stage': {'algorithmic_bytes': stage_bytes, 'ms': ms,
                               'frac': stage_bytes / (ms * 1e-3) / 1e9 / peak,
                               'what': 'SURVEY 8d bytes of the whole step on this rank (text in, normalized text, ids / ends, row '
                                       'offsets) over its device time'}},
        'cpu_baseline': cpu, 'clocks': clocks,
    }


def config1_latency(reps, dump=None):
    """BASELINE.json configs[0]: `aksharTokenizer().tokenize(line)` (no model: akshar-level fallback) over the reference's
    data/corpus.txt, one string per call -- the latency of the drop-in API (each call: pinned staging, two library calls,
    read-back), next to the same lines as ONE batch and to the CPU port of the same function on this box.  BASELINE.md
    quotes 62 us/line for the reference's own Python path.  With `dump`, the akshars of the last pass are added to it."""
    import numpy as np
    import torch
    import akshar_b200 as A
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import akshar_oracle as O
    with open(os.path.join(ROOT, 'tests', 'golden', 'corpus.txt'), encoding='utf-8') as f:
        lines = [ln.strip() for ln in f.readlines() if ln.strip()]
    tk = A.aksharTokenizer()
    exp = [O.segment_akshars(O.normalize_text(s)) for s in lines]
    assert [tk.tokenize(s) for s in lines] == exp and tk.tokenize_batch(lines) == exp
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        last = [tk.tokenize(s) for s in lines]
    one = (time.perf_counter() - t0) / (reps * len(lines))
    if dump is not None:
        flat = [a for row in last for a in row]
        dump['latency_akshars_per_line'] = np.array([len(row) for row in last], dtype=np.float64)
        dump['latency_akshar_lengths'] = np.array([len(a) for a in flat], dtype=np.float64)
        dump['latency_akshar_code_points'] = np.array([ord(c) for a in flat for c in a], dtype=np.float64)
    t0 = time.perf_counter()
    for _ in range(reps):
        tk.tokenize_batch(lines)
    batch = (time.perf_counter() - t0) / (reps * len(lines))
    t0 = time.perf_counter()
    for _ in range(reps):
        for s in lines:
            O.segment_akshars(O.normalize_text(s))
    cpu = (time.perf_counter() - t0) / (reps * len(lines))
    nbytes = sum(len(s.encode('utf-8')) for s in lines)
    return {'metric': 'us_per_line_tokenize_single_string', 'value': one * 1e6, 'unit': 'us/line', 'higher_is_better': False,
            'config': {'workload': 'configs[0]: aksharTokenizer().tokenize(line), akshar-level fallback, %d lines / %d bytes of '
                                   'data/corpus.txt, one string per call' % (len(lines), nbytes)},
            'same_lines_as_one_batch_us_per_line': batch * 1e6, 'parity_in_run': True, 'rows_compared': len(lines),
            'cpu_baseline': {'value': cpu * 1e6, 'unit': 'us/line', 'cores': 1, 'kind': 'port',
                             'sample': 'oracle normalize_text + segment_akshars, same lines, %d passes' % reps},
            'reference_published_us_per_line': 62.0,
            'note': 'a single short string is launch- and read-back-latency bound on any GPU path; the batch entry points are the product'}


# ------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--mb', type=int, default=None, help='synthetic input per GPU in MiB (default: the configuration the metric is quoted on)')
    ap.add_argument('--workload', default=None, choices=['bpe', 'unigram', 'pipeline', 'mixed'])
    ap.add_argument('--cpu-sample-mb', type=float, default=24.0)
    ap.add_argument('--no-also', action='store_true', help='headline workload only')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed step computed (a seeded sample of rows) as DIR/<name>.npy')
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    dump = {} if a.dump_outputs else None
    R = Rank()
    workload = a.workload or ('bpe' if R.world == 1 else 'mixed')
    mb = a.mb or {'bpe': 1024, 'unigram': 1024, 'pipeline': 4096, 'mixed': 4096}[workload]

    if a.impl == 'reference':
        if R.rank != 0:
            return
        sample = int(a.cpu_sample_mb * (1 << 20))
        data, off = make_corpus(KIND[workload], sample + (1 << 20), 0)
        arm = CpuArm(workload, data, off, sample)
        for _ in range(a.warmup):
            arm.step()
        t = tok = 0.0
        for _ in range(a.steps):
            dt, n = arm.step()
            t += dt
            tok += n
        native = arm.native_libs()
        arm.close()
        if dump is not None:
            import numpy as np
            # what the CPU arm returns: one checksum of the reference's output per row of the sample
            write_dump(a.dump_outputs, {'reference_%s_row_checksums' % workload: np.array(arm.sums, dtype=np.float64)})
        v = arm.nbytes * a.steps / t / 1e9
        metric = 'utf8_input_GBps_batch_encode' if workload != 'pipeline' else 'utf8_input_GBps_normalize_segment'
        print(json.dumps({
            'impl': 'reference', 'metric': metric, 'value': v, 'unit': 'GB/s', 'tokens_per_s': tok / t, 'n_gpus': a.gpus,
            'steps': a.steps, 'warmup': a.warmup, 'ms_per_step': t / a.steps * 1e3, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'u8', 'data': 'synthetic',
            'config': {'workload': describe(workload, mb, R.world), 'bytes_per_gpu': mb << 20},
            'cpu_baseline': {'value': v, 'unit': 'GB/s', 'cores': arm.cores, 'kind': 'port',
                             'sample': '%d rows / %.1f MB of the same synthetic workload per step; oracle/akshar_oracle.py '
                                       '(pure-Python restatement; the reference itself is Python and cannot travel to this box)'
                                       % (len(arm.lines), arm.nbytes / 1e6),
                             'native_libs_alone': native},
            'e2e': {'value': v, 'unit': 'GB/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}))
        return

    import torch
    dist = None
    torch.cuda.set_device(R.local)
    if R.world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=torch.device('cuda', R.local))
    from akshar_b200 import _lib
    _lib.load()                 # the library __graft_entry__.build() compiled; nothing is compiled here
    line = run_workload(R, workload, mb, a.steps, a.warmup, a.cpu_sample_mb, dist, dump=dump)
    if a.workload is None and R.world == 1 and not a.no_also:
        # BASELINE.json configs[2] and configs[3], measured the same way (smaller CPU samples)
        import gc
        also = []
        for w, wmb in (('unigram', 1024), ('pipeline', 4096)):
            gc.collect()
            torch.cuda.empty_cache()
            also.append(run_workload(R, w, wmb, a.steps, a.warmup, min(a.cpu_sample_mb, 8.0), dist, dump=dump))
        also.append(config1_latency(a.steps, dump))
        line['also'] = also
    if R.rank == 0:
        if dump is not None:
            write_dump(a.dump_outputs, dump)
        print(json.dumps(line))
    if R.world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
