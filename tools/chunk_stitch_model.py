"""CPU model of the general chunk walk (empty matches, slice emulation) + stitch_check, with and
without a candidate fix for the known gap of DESIGN.md section 2 (re-derive the first span's
start with slice_start at the real entry point).  Usage: python tools/chunk_stitch_model.py SEED SECONDS

Round-1 finding (tiny 8/24-byte chunks, random look-around patterns): the current rule is wrong in
~1.4 % of cases; the candidate fix removes ~90 % of them but not all (matches whose slice-rule
start is no true match start need the walk itself to apply the rule at speculative entries).
Two things are needed for exactness: (1) the first span of an accepted speculative chunk gets its
start from slice_start(real entry, end) -- the candidate fix modelled here -- and (2) a chunk
without matches must hand on the restart point it RECEIVED, not the one it assumed (its own first
position); (2) is a "last chunk with matches" prefix propagation over runs of empty chunks and is
what the remaining ~10 % are.  Patterns without look-arounds are unaffected
(tests/test_stitch_trim_sim.py, shard fuzz)."""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
import numpy as np
import regex_b200 as R
from dfa_sim import Sim
from oracle import oracle as O
from helpers import xorshift_bytes
import test_fuzz_tables_vs_oracle as F
SPEC="spec"
def walk(sim, S, text, k, chunk, p, lm, chain, emulate, utf8=False):
    n=len(text); cb, ce = k*chunk, min((k+1)*chunk, n)
    spans=[]; fc=None
    while p is not None:
        lo=max(p, cb+1)
        if k==0 and p==0 and S[0]: s=0
        else: s=next((q for q in range(lo, ce+1) if S[q]), None)
        if s is None: break
        if fc is None: fc=s
        e=sim.anchored_end(text, s)
        ms=s
        if emulate and chain and e!=p:
            ms=sim.slice_start(text, p, e)
            if ms is None: p=None; break
        chain=True
        if ms==e:
            p=sim.next_after_empty(text, e)
            if e==lm: continue
        else: p=e
        lm=e
        spans.append((ms,e))
    return spans, p, lm, fc
def chunked(sim, text, chunk, fix):
    info=sim.info; emulate=info["has_looks"]; cme=info["can_match_empty"]
    n=len(text); S=sim.start_bitmap(text)
    nc=max(1,(n+chunk-1)//chunk)
    st=[]; in_p=[0]+[SPEC]*(nc-1); in_lm=[None]*nc
    for k in range(nc):
        if k==0: spans,p,lm,fc=walk(sim,S,text,0,chunk,0,None,True,emulate)
        else: spans,p,lm,fc=walk(sim,S,text,k,chunk,k*chunk+1,None,False,emulate)
        st.append(dict(spans=spans,out_p=p,out_lm=lm,fc=fc))
    for _ in range(4*nc+8):
        outs=[(s["out_p"],s["out_lm"]) for s in st]; dirty=[]
        for k in range(1,nc):
            tp,tl=outs[k-1]; cp=in_p[k]; c_first=k*chunk+1
            if cp==SPEC:
                if tp is None: ok=False
                elif emulate or cme: ok = tp < c_first or (tp==c_first and not emulate and not (cme and tl==c_first))
                else: ok = (st[k]["fc"] is None or tp<=st[k]["fc"]) and tp<=c_first+chunk
                if ok and fix and emulate and st[k]["spans"]:
                    # proposed fix: the first span's start under the slice rule at the real entry
                    s0,e0=st[k]["spans"][0]
                    if e0!=tp:
                        ms=sim.slice_start(text,tp,e0)
                        if ms is None or (ms==e0)!=(s0==e0): ok=False
                        elif ms!=s0: st[k]["spans"][0]=(ms,e0)
            else: ok = (cp,in_lm[k])==(tp,tl)
            if not ok:
                in_p[k]=tp; in_lm[k]=tl; dirty.append(k)
        for k in dirty:
            spans,p,lm,fc=walk(sim,S,text,k,chunk,in_p[k],in_lm[k],True,emulate)
            st[k]=dict(spans=spans,out_p=p,out_lm=lm,fc=fc)
        if not dirty: break
    out=[]
    for s in st: out+=s["spans"]
    # the iteration may have ended inside a chunk (p None): later chunks' spans are void
    res=[]; 
    for k,s in enumerate(st):
        res+=s["spans"]
        if s["out_p"] is None: break
    return res
rng=np.random.Generator(np.random.PCG64(int(sys.argv[1]))); t0=time.time(); n=0; bad={False:0,True:0}
while time.time()-t0<float(sys.argv[2]):
    p=F._pattern(rng)
    try: r=R.BytesRegex("(?-u)"+p if "α" not in p and "é" not in p and "3b1" not in p and "pL" not in p else p)
    except R.Error: continue
    sim=Sim(r)
    if not sim.info["has_looks"]: continue
    o=O.OracleRegex(r._pattern if hasattr(r,"_pattern") else ("(?-u)"+p if "α" not in p and "é" not in p and "3b1" not in p and "pL" not in p else p))
    for seed in (1,2):
        text=xorshift_bytes(int(rng.integers(0,999)), 150, b"abc \n")
        exp=o.find_iter(text)
        for chunk in (8,24):
            n+=1
            for fix in (False,True):
                try: got=chunked(sim,text,chunk,fix)
                except AssertionError: got="ASSERT"
                if got!=exp:
                    bad[fix]+=1
                    if fix and bad[True]<=5: print("STILL BAD with fix", repr(p), chunk, str(got)[:80], exp[:5])
print("cases",n,"bad without fix",bad[False],"bad with fix",bad[True])
