"""One MIDA launch per configuration, for ncu captures: python tools/mida_once.py [n]"""
import sys
from pathlib import Path
import torch
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from invesalius3_b200 import projection

n = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
g = torch.Generator(device="cuda").manual_seed(0)
vol = torch.randint(-1024, 3072, (n, n, n), dtype=torch.int16, device="cuda", generator=g)
for axis in (0, 2):
    o = projection.mida(vol, axis, 32000, 2)        # opacity 0: every ray walks the whole volume
    o = projection.mida(vol, axis, 1000, 4000)      # opacity ramp: per-sample division, late exit
torch.cuda.synchronize()
print("ok")
