import sys, json, torch, numpy as np
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from scipy.ndimage import generate_binary_structure
from invesalius3_b200 import _lib, device as dev, phantom
lib=_lib.load()
vol=phantom.ct((512,512,512),seed=2); seed=phantom.first_seed_in_range(vol,256,226,3071)
t=torch.from_numpy(vol).cuda(); st=generate_binary_structure(3,1)
ref=None
for eng in (0,1,0,1):
    lib.b2v_floodfill_set_engine(eng)
    out=torch.zeros(vol.shape,dtype=torch.uint8,device='cuda')
    for _ in range(3): out.zero_(); dev.floodfill_threshold(t,[seed],226,3071,254,st,out)
    ts=[]
    for _ in range(10):
        out.zero_(); a=torch.cuda.Event(enable_timing=True); b=torch.cuda.Event(enable_timing=True)
        a.record(); stt={}; r=dev.floodfill_threshold(t,[seed],226,3071,254,st,out,stats=stt); b.record(); torch.cuda.synchronize(); ts.append(a.elapsed_time(b))
    if ref is None: ref=out.clone()
    print("engine",eng,"rounds",r,"median ms",sorted(ts)[5],"min",min(ts),"equal",bool(torch.equal(ref,out)),"filled",int((out==254).sum()),stt)
st26=generate_binary_structure(3,3)
for eng in (0,1):
    lib.b2v_floodfill_set_engine(eng)
    out=torch.zeros(vol.shape,dtype=torch.uint8,device='cuda')
    ts=[]
    for _ in range(5):
        out.zero_(); a=torch.cuda.Event(enable_timing=True); b=torch.cuda.Event(enable_timing=True)
        a.record(); r=dev.floodfill_threshold(t,[seed],226,3071,254,st26,out); b.record(); torch.cuda.synchronize(); ts.append(a.elapsed_time(b))
    print("26-conn engine",eng,"rounds",r,"median ms",sorted(ts)[2],"filled",int((out==254).sum()))
