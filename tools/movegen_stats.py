"""Search statistics of the movegen sweep's kernel (needs a build with TRL_NVCC_EXTRA=-DTRL_MOVEGEN_STATS):
python tools/movegen_stats.py.  Runs the pass form, as the sweep does: rounds, fill iterations, (rotation, direction)
passes and kick tests are those of the specialised closure search in movegen_rows_kernel and, for the T searches it
deferred, once more in movegen_t_order_kernel; a pair of twin passes packed into one word counts as one pass.  The first
line mixes two piece types per call, so it also counts the searches the legacy route repeats for the other piece of an
undecided call; the per-piece lines search one piece per call (the T line counts a deferred search twice)."""
import ctypes, sys, os
import numpy as np, torch
sys.path.insert(0, os.getcwd())
from tetris_reinforcement_learning_b200 import _native, move_generation, synth
from tetris_reinforcement_learning_b200.const import MASK_WORDS
L=_native.lib(); L.trl_movegen_warp_form(2)
dev=torch.device("cuda:0")
boards,cur,alt=synth.movegen_workload(20000)
n=boards.shape[0]
d_b=torch.from_numpy(boards.view(np.int16)).to(dev); d_c=torch.from_numpy(cur).to(dev); d_a=torch.from_numpy(alt).to(dev)
d_mask=torch.zeros((n,MASK_WORDS),dtype=torch.int32,device=dev); d_n=torch.zeros(n,dtype=torch.int16,device=dev); d_st=torch.zeros(n,dtype=torch.int32,device=dev)
st=(ctypes.c_uint64*16)()
L.trl_debug_movegen_fast_stats(st)
move_generation.movegen_device(d_b,d_c,d_a,d_mask,None,d_n,d_st); torch.cuda.synchronize()
L.trl_debug_movegen_fast_stats(st)
s=[int(x) for x in st]; tot=s[0]+s[1]
print("searches",tot,"fallback %.3f%%"%(100*s[1]/tot),"rounds/search %.2f fill iters %.2f kd passes %.2f kick tests %.2f"%(s[2]/tot,s[3]/tot,s[4]/tot,s[5]/tot))
# by piece type of cur (alt varies): run single-piece calls
for t in range(7):
    c=np.full(n,t,np.uint8)
    d_c2=torch.from_numpy(c).to(dev)
    move_generation.movegen_device(d_b,d_c2,d_c2,d_mask,None,d_n,d_st); torch.cuda.synchronize()
    L.trl_debug_movegen_fast_stats(st); s=[int(x) for x in st]; tot=s[0]+s[1]
    print("piece",t,"searches",tot,"fallback %.3f%%"%(100*s[1]/tot),"rounds %.2f fill iters %.2f kd passes %.2f kick tests %.2f"%(s[2]/tot,s[3]/tot,s[4]/tot,s[5]/tot), "placements/search %.1f"%(float(d_n.to(torch.int64).sum())/n), "mixed after round 1: %.3f%% of searches"%(100*s[6]/tot),
          "| order analysis: no edges %d, C1 %d, C2 %d, cells reached later %d, seed cells %d, late/level-2 conflict %d, undecided %d, decided %d"%tuple(s[8:16]))
