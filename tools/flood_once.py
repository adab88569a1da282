import sys, torch
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from scipy.ndimage import generate_binary_structure
from invesalius3_b200 import device as dev, phantom
vol = phantom.ct((512, 512, 512), seed=2); seed = phantom.first_seed_in_range(vol, 256, 226, 3071)
t = torch.from_numpy(vol).cuda(); st = generate_binary_structure(3, 1)
out = torch.zeros(vol.shape, dtype=torch.uint8, device='cuda')
for _ in range(3):
    out.zero_(); stt = {}; r = dev.floodfill_threshold(t, [seed], 226, 3071, 254, st, out, stats=stt)
torch.cuda.synchronize(); print(r, stt)
from invesalius3_b200 import _lib
import ctypes as C
lay=(C.c_int64*8)(); _lib.call('b2v_floodfill_layout',512,512,512,1,lay)

