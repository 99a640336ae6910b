"""Per-phase clock stamps of CTA 0's third work item in the x3 backward at cfg2 size (--cache: the variant that loads the
forward's chunk cache; its stamps 1-3 coincide)."""
import ctypes, os, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import wkv7 as O
import visualrwkv_b200.wkv7 as W
from visualrwkv_b200 import _lib
names = ["wait_in+P1", "mma_scores", "P2", "inverse(+mmaB4)", "wait_dS", "dZ+C1", "P3+C2(+Upair)", "P4+S0", "C3+P5", "D batch", "P6", "D3b/D4b", "epilogue"]
dbg = torch.zeros(4096, dtype=torch.float32, device="cuda")
_lib.check(_lib.lib().vrwkv_wkv7_chunk_debug(ctypes.c_void_p(dbg.data_ptr())), "dbg")
B, T, H = 8, 2048, 12
w, q, k, v, a, b, dy = [x.cuda() for x in O.make_inputs(B, T, H, 64, seed=42)]
cache = None
if "--cache" in sys.argv:
    y, s, sa, cache = W.forward_raw(w, q, k, v, a, b, bounded_decay=True, chunk_checkpoints=True, chunk_cache=True)
else:
    y, s, sa = W.forward_raw(w, q, k, v, a, b, bounded_decay=True, chunk_checkpoints=True)
dbg.zero_()
W.backward_raw(w, q, k, v, a, b, dy, s, sa, bounded_decay=True, cache=cache)
torch.cuda.synchronize()
ts = [int(x) for x in dbg.cpu().numpy()[3072:3072 + 14]]
d = [ts[i + 1] - ts[i] for i in range(13)]
print("total", ts[13], " ".join(f"{n}={x}" for n, x in zip(names, d)))
_lib.check(_lib.lib().vrwkv_wkv7_chunk_debug(ctypes.c_void_p(0)), "dbg")
