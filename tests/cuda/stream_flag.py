"""FE_GEMM_TRACE build only: which bounded wait of the streaming kernel timed out (code * 1000 + warp)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ctypes as C
import numpy as np, torch
import b200_frontend as fe
import helpers
m = fe.LFCCDelta(**helpers.LFCC_CFG, variant="dft_gemm")
eng = m.engine
R = int(sys.argv[1]) if len(sys.argv) > 1 else 8
x = (0.1 * torch.randn(R, 64600, device="cuda")).clamp_(-1, 1)
try:
    e = eng.fbank_energies(x)
    torch.cuda.synchronize()
    print("ok")
except Exception as ex:
    print("error:", str(ex)[:100])
ws = eng._workspace[x.device][torch.cuda.current_stream().cuda_stream]   # the current stream's workspace
nbytes = eng.lib.b200fe_workspace_bytes(C.byref(eng.params), R, 64600)
try:
    tail = ws[nbytes - 65536: nbytes - 65536 + 16].cpu().numpy()
    print("flag", tail.view(np.int32)[:4])
except Exception as ex:
    print("could not read flag:", str(ex)[:100])
