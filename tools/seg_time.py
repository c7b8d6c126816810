import os, sys, time
ROOT=os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0]=[ROOT,os.path.join(ROOT,'tools')]
import torch, akshar_b200 as A, synth_corpus as sc
eng=A.Engine(0)
d,o=sc.Corpus('social',20261018).generate(1<<30)
b=eng.put((torch.from_numpy(d),torch.from_numpy(o)))
norm=eng.normalize_batch(b)
for name,kw in (('clusters+runs',dict(clusters=True,runs=True)),('clusters',dict(clusters=True,runs=False))):
    for _ in range(2): eng.segment_batch(norm, check=False, **kw)
    torch.cuda.synchronize()
    e0,e1=torch.cuda.Event(enable_timing=True),torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5): eng.segment_batch(norm, check=False, **kw)
    e1.record(); torch.cuda.synchronize()
    print('segment offsets', name, e0.elapsed_time(e1)/5, 'ms per GiB')
    for _ in range(2): eng.segment_masks(norm, check=False, **kw)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(5): eng.segment_masks(norm, check=False, **kw)
    e1.record(); torch.cuda.synchronize()
    print('segment masks  ', name, e0.elapsed_time(e1)/5, 'ms per GiB')
