import os, sys, numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tools'))
import regex_b200 as R, corpus as C
SEG=3584; L=32
text = np.frombuffer(bytes(C.host_corpus(SEG*L*4)), dtype=np.uint8)
def run(pat, strides):
    r = R.BytesRegex(pat)
    d = r.dfa(1)
    trans, classes, start, match_lo = d["trans"], d["classes"], d["start"], d["match_lo"]
    n_states = trans.shape[0]
    nxt = trans[:, classes[np.arange(256)]]
    ids = np.zeros(n_states, dtype=np.int64); k=2
    for s in range(1,n_states):
        if s < match_lo: ids[s]=k; k+=1
    m=0
    for s in range(match_lo, n_states):
        m+=1; ids[s]=-m
    # precompute state/byte sequences
    seqs=[]
    for blk in range(2):
        segs = text[blk*SEG*L:(blk+1)*SEG*L].reshape(L,SEG)
        st = np.full(L, start[32], dtype=np.int64)
        for j in range(SEG-1,-1,-1):
            b = segs[:,j].astype(np.int64)
            seqs.append((st.copy(), b))
            st = nxt[st, b]
    out={}
    for stride in strides:
        tot=0
        for st,b in seqs:
            words = ids[st]*stride + (b>>2)
            u = np.unique(words)
            tot += np.bincount(u & 31, minlength=32).max()
        out[stride]=round(tot/len(seqs),3)
    print(pat, "states", n_states, out)
strides=[64,65,66,67,68,69,70,71,72,73,74,76,78,80]
for p in sys.argv[1:]: run(p, strides)
