import numpy as np, torch, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import oracle
from ronkathon_b200 import Context, ops
torch.cuda.set_device(0)
ctx=Context(0, torch.cuda.current_stream().cuda_stream)
GL=oracle.GOLDILOCKS
d=ops.splitmix_fill(ctx,1<<24,42,GL,'cuda')
a=ops.to_host(d)
ops.ntt_(ctx,d,24); ctx.sync()
X=ops.to_host(d)
w=oracle.root_of_unity(GL,1<<24)
print("spots", [int(X[k])==oracle.poly_eval_horner(GL,a,pow(w,k,GL)) for k in (0,1,5,(1<<23)+3,(1<<24)-1)])
ops.ntt_(ctx,d,24,inverse=True); ctx.sync()
print("roundtrip", bool(np.array_equal(ops.to_host(d),a)))
