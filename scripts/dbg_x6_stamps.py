"""Per-phase clock stamps of CTA 0's third work item in the x6 forward at cfg2 size."""
import ctypes, os, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import wkv7 as O
import visualrwkv_b200.wkv7 as W
from visualrwkv_b200 import _lib
names = ["wait_in", "P1", "mma_scores", "P2", "inverse(+mmaAV)", "P3", "mma_W", "P4", "mma_CORR", "P5", "wait_state", "S0parts", "mma_UY", "P7", "mma_Z", "P8+flag"]
dbg = torch.zeros(4096, dtype=torch.float32, device="cuda")
_lib.check(_lib.lib().vrwkv_wkv7_chunk_debug(ctypes.c_void_p(dbg.data_ptr())), "dbg")
B, T, H = 8, 2048, 12
w, q, k, v, a, b, dy = [x.cuda() for x in O.make_inputs(B, T, H, 64, seed=42)]
for ck, cache in ((True, False), (False, False), (True, True)):
    W.set_variant(6, 0)
    dbg.zero_()
    W.forward_raw(w, q, k, v, a, b, bounded_decay=True, chunk_checkpoints=ck, chunk_cache=cache)
    torch.cuda.synchronize()
    ts = [int(x) for x in dbg.cpu().numpy()[2048:2048 + 17]]
    d = [ts[i + 1] - ts[i] for i in range(16)]
    print("ck64+cache" if cache else "ck64" if ck else "ck16", "total", ts[16], " ".join(f"{n}={x}" for n, x in zip(names, d)))
W.set_variant(0, 0)
_lib.check(_lib.lib().vrwkv_wkv7_chunk_debug(ctypes.c_void_p(0)), "dbg")
