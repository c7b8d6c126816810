#!/usr/bin/env python
"""What the words that are new in a call cost: the resolve kernel with the word cache restored at every call (default) and held."""
import sys, os
ROOT=os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0]=[ROOT,os.path.join(ROOT,'tools')]
import torch, akshar_b200 as A, synth_corpus as sc
for what,kind,model,k in (('unigram','hindi','spm24k.model',1),('bpe','hinglish','bpe24k.json',0)):
    tk=A.aksharTokenizer(os.path.join(ROOT,'tests','golden','models',model), 'sentencepiece' if k else 'bpe')
    eng=tk._eng
    d,o=sc.Corpus(kind,20261018).generate(1<<30)
    b=eng.put((torch.from_numpy(d),torch.from_numpy(o)))
    name='ak_resolve_kernel<%s>'%what
    for hold in (0,1):
        eng.lib.akshar_word_cache_hold(eng._h, hold)
        eng.timing(True)
        ts=[]
        for _ in range(4):
            eng.tokenizer_encode_batch(b,k,check=False); torch.cuda.synchronize()
            ts.append(eng.kernel_ms(name))
        eng.timing(False)
        print(what,'hold',hold,'resolve ms per step:',['%.2f'%t for t in ts])
