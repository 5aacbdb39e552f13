"""Scratch experiment kept for the record: back-to-back launches on ROTATING buffers (so that no input is L2-resident)
for the flat forward / backward kernels at several sizes - the source of the "rotating buffers" figures quoted in the
round-1 kernel history.   python profiles/tail_experiment.py"""
import ctypes as C, math, sys, torch
sys.path.insert(0, "/root/repo")
from dlmc_quant_b200 import _lib, functional as F
h=_lib.lib()
def run(n, nbuf=24, iters=240):
    nbuf = max(2, min(nbuf, int(3e9 // (n * 12)))); iters = nbuf * 6
    xs=[torch.relu(torch.randn(n,device="cuda")) for _ in range(nbuf)]
    dys=[torch.randn(n,device="cuda") for _ in range(nbuf)]
    ys=[torch.empty(n,device="cuda") for _ in range(nbuf)]
    scale=torch.full((1,),0.2,device="cuda"); off=torch.zeros(1,device="cuda"); ds=torch.zeros(1,device="cuda")
    lay=_lib.Layout(1,1,n,0); qp=_lib.QParams(1,0,15,1e-4,scale.data_ptr(),off.data_ptr())
    wsn=h.dlmcq_workspace_bytes(None); ws=torch.zeros(wsn,dtype=torch.uint8,device="cuda")
    cur=lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)
    def fwd(i): h.dlmcq_fq_forward(xs[i].data_ptr(), ys[i].data_ptr(), None, C.byref(lay), C.byref(qp), cur())
    def bwd(i): h.dlmcq_fq_backward(xs[i].data_ptr(), dys[i].data_ptr(), ys[i].data_ptr(), ds.data_ptr(), None, C.byref(lay), C.byref(qp), ws.data_ptr(), wsn, cur())
    out=[]
    for f in (fwd,bwd):
        g=torch.cuda.CUDAGraph()
        for i in range(nbuf): f(i)
        torch.cuda.synchronize()
        with torch.cuda.graph(g):
            for k in range(iters): f(k%nbuf)
        g.replay(); torch.cuda.synchronize()
        a,b=torch.cuda.Event(enable_timing=True),torch.cuda.Event(enable_timing=True)
        a.record(); g.replay(); b.record(); torch.cuda.synchronize()
        out.append(a.elapsed_time(b)*1e3/iters)
    return out
for n in [int(a) for a in sys.argv[1:]] or (1605632, 3211264, 6422528, 12845056):
    f,b=run(n)
    print(f"n={n}: fwd {f:.2f} us ({8*n/f/1e3:.0f} GB/s)  bwd {b:.2f} us ({12*n/b/1e3:.0f} GB/s)")
