"""FE_GEMM_TRACE build only: dump the SM-clock timeline of CTA 0's pipeline events."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ctypes as C
import numpy as np, torch
import b200_frontend as fe
import helpers
m = fe.LFCCDelta(**helpers.LFCC_CFG, variant="dft_gemm")
eng = m.engine
R = 592
x = (0.1 * torch.randn(R, 64600, device="cuda")).clamp_(-1, 1)
for _ in range(2):
    e = eng.fbank_energies(x)
torch.cuda.synchronize()
ws = eng._workspace[x.device][torch.cuda.current_stream().cuda_stream]   # the current stream's workspace
nbytes = eng.lib.b200fe_workspace_bytes(C.byref(eng.params), R, 64600)
tail = ws[nbytes - 65536: nbytes].cpu().numpy()
tr = np.frombuffer(tail[256:256 + 8 * 8 * 16 * 8].tobytes(), dtype=np.int64).reshape(8, 8, 16)
base = tr[0, 0, 0]
names = ["ld_issue", "samp_full", "a_full_arr", "mma_issue", "acc_full", "acc_empty_arr", "epi_done", "mma_tile_start"]
for it in range(6):
    print("tile", it)
    for q in range(5):
        print("  q", q, {names[e]: int(tr[it, q, e] - base) for e in range(4)})
    print("   ", {names[e]: int(tr[it, 0, e] - base) for e in range(4, 8)})
    print("    scout start/done, producer got scout:", [int(tr[it, 0, e] - base) for e in (10, 11, 12)])
    print("    epi chunks (after ld wait, after bins):", [(int(tr[it, c, 8] - base), int(tr[it, c, 9] - base)) for c in range(4)])
