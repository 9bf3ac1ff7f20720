"""Hand-off timeline of the S-store similarity kernel's first tiles (debug build with -DCOR_SIM_TRACE, see sim_umma.cu):
COR_B200_LIB=cor_b200/build/ab/libcor_b200_trace.so python benchmarks/sim_trace.py [Nq Nr]"""
import ctypes as C
import os
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from cor_b200 import _lib as L, ops
Nq, Nr = (int(sys.argv[1]), int(sys.argv[2])) if len(sys.argv) > 2 else (1024, 102400)
g = torch.Generator(device="cuda").manual_seed(0)
R = torch.nn.functional.normalize(torch.randn(Nr, 256, device="cuda", generator=g), dim=-1).bfloat16()
Q = torch.nn.functional.normalize(torch.randn(Nq, 256, device="cuda", generator=g), dim=-1).bfloat16()
for _ in range(3):
    ops._sim_forward(R, Q, 1.0, True, False, "umma")
torch.cuda.synchronize()
lib = L.load()
buf = (C.c_longlong * 256)()
lib.cor_debug_sim_trace.restype = C.c_int
assert lib.cor_debug_sim_trace(buf) == 0
t0 = min(v for v in buf if v > 0)
names = ["mma_start", "mma_issued", "epi_accfull", "epi_release", "epi_done", "tma_issued"]
print("tile " + " ".join(f"{n:>12}" for n in names))
for t in range(24):
    row = [buf[t * 8 + e] for e in range(6)]
    print(f"{t:4d} " + " ".join(f"{(v - t0) if v > 0 else -1:12d}" for v in row))
