import os, sys, time; sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import numpy as np, scipy.sparse as sp
from proto_pc import *
for nx in (128,256,512):
    m = M.create_unit_square(None, nx, nx)
    class P: pass
    prob=P(); prob.x=m.geometry.x[:,:2]; prob.cells=m.geometry.dofmap; prob.n=prob.x.shape[0]
    L,ml=laplace_mass(prob); n=prob.n
    Lr=(L+1e-8*sp.diags(ml)).tocsr()
    rb=np.random.default_rng(1).standard_normal(n); rb-=rb.mean()
    for over in (1.0,1.5,1.8):
        t0=time.time()
        amg=AMG(Lr,L,1,theta=0.0,smoother='cheb',over=over,cheb_deg=3)
        x,its,res=fgmres(Lr,rb,lambda r: amg.vcycle(r),rtol=1e-6,maxit=200)
        x,its2,res=fgmres(Lr,rb,lambda r: amg.vcycle(r),rtol=1e-2,maxit=200)
        print(f'nx {nx} over {over}: its(1e-6) {its} its(1e-2) {its2}  t {time.time()-t0:.1f}')
