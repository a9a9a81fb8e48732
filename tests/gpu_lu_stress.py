"""Development driver (not a pytest file): 750 strict-build runs of the warp-per-circuit LU (n = 1..8, 257 systems) against
the oracle with the device allocator dirtied by NaN-filled buffers in between — hunts for reads of uninitialised memory."""
import numpy as np, torch
import parity_util as PU
from test_lu_operator import mna_like
T,O=PU.T,PU.O
ctx=T.Context(0)
bad=0
# dirty the allocator: fill and free large device buffers with NaN patterns
for it in range(150):
    junk=torch.full((64*1024*1024//8,), float('nan'), dtype=torch.float64, device='cuda'); del junk
    torch.cuda.empty_cache()
    for n in (1,2,3,5,8):
        n_inst=257
        base,A,b=mna_like(n,n_inst,7*n+it)
        order=T.lu_order(base)
        x,st=ctx.lu_solve_batched(A,b,order,strict=True)
        xo,sto,_=O.lu_batch(base,A,b)
        if not (np.array_equal(st,sto) and np.array_equal(x,xo)):
            bad+=1
            k=np.nonzero((st!=sto)|np.any(x!=xo,axis=1))[0]
            print("MISMATCH it",it,"n",n,"inst",k[:8],"st",st[k[:4]],"x",x[k[:2]],"xo",xo[k[:2]],flush=True)
print("done, mismatches:",bad)
