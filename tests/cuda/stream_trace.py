"""FE_GEMM_TRACE build only (make LIBDIR=../lib_trace EXTRA_NVFLAGS=-DFE_GEMM_TRACE; B200FE_LIB=...): SM-clock
timeline of CTA 0 of the streaming kernel."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ctypes as C
import numpy as np, torch
import b200_frontend as fe
import helpers
m = fe.LFCCDelta(**helpers.LFCC_CFG, variant="dft_gemm")
eng = m.engine
R = int(sys.argv[1]) if len(sys.argv) > 1 else 1184
N = int(sys.argv[2]) if len(sys.argv) > 2 else 4     # launches before the traced (last) one: a long run shows the sustained state
x = (0.1 * torch.randn(R, 64600, device="cuda")).clamp_(-1, 1)
t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
for i in range(N):
    if i == N - 1:
        t0.record()
    e = eng.fbank_energies(x)
t1.record()
torch.cuda.synchronize()
print("last launch: %.3f ms" % t0.elapsed_time(t1))
ws = eng._workspace[x.device][torch.cuda.current_stream().cuda_stream]   # the current stream's workspace
nbytes = eng.lib.b200fe_workspace_bytes(C.byref(eng.params), R, 64600)
tail = ws[nbytes - 65536: nbytes].cpu().numpy()
print("flag", tail[:4].view(np.int32)[0])
tr = np.frombuffer(tail[256:256 + 8 * 8 * 16 * 8].tobytes(), dtype=np.int64).reshape(8, 8, 16)
base = tr[0, 0, 0]
for it in range(7):
    r = lambda q, e: int(tr[it, q, e] - base)
    print("tile", it, "loader_start", r(0, 0), "edges_done", r(0, 9), "samp_full", r(0, 1), "scout_done", r(0, 7), "acc_empty_seen", r(0, 8))
    print("    b_full(q):", [r(q, 10) for q in range(5)], " mma_issue(q):", [r(q, 3) for q in range(5)], " produced(q):", [r(q, 2) for q in range(5)])
    print("    drain run0/1: acc_full", r(0, 4), r(1, 4), "walk_done", r(0, 5), r(1, 5), "tile_done", r(0, 6), r(1, 6))
