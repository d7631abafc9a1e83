import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tools'))
import torch, corpus as C, regex_b200 as R
dev=torch.device("cuda",0)
text=C.device_corpus(1<<30, C.SEED, dev)
r=R.BytesRegex(r"[a-zA-Z]+ing"); r.set_fuse(False)
n=r.find_all_device(text)
out=torch.empty((n+16,2),dtype=torch.int64,device=dev)
for _ in range(2): r.find_all_device(text,out)
