import ctypes as C, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
torch.cuda.init(); torch.zeros(1,device='cuda')
from vittracker_b200 import _lib
lib=_lib.load()
out=(C.c_int*10)()
lib.vt_debug_fused_occupancy(out)
print(list(out))
