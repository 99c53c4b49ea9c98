"""FE_GEMM_TRACE build: run one small launch and print the barrier-timeout flag (code*1000 + warp)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ctypes as C
import numpy as np, torch
import b200_frontend as fe
import helpers
m = fe.LFCCDelta(**helpers.LFCC_CFG, variant="dft_gemm")
eng = m.engine
R = int(sys.argv[1]) if len(sys.argv) > 1 else 2
x = (0.1 * torch.randn(R, 64600, device="cuda")).clamp_(-1, 1)
e = eng.fbank_energies(x)
torch.cuda.synchronize()
ws = eng._workspace[x.device][torch.cuda.current_stream().cuda_stream]   # the current stream's workspace
nbytes = eng.lib.b200fe_workspace_bytes(C.byref(eng.params), R, 64600)
flag = ws[nbytes - 65536: nbytes - 65536 + 4].cpu().numpy().view(np.int32)[0]
print("timeout flag:", flag, "(0 = none; else code*1000 + warp)")
print("finite:", bool(torch.isfinite(e).all()), "max", float(e.max()))
