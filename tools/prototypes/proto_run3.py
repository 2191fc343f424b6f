import os, sys, time; sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import numpy as np, scipy.sparse as sp, scipy.sparse.linalg as spla
from proto_pc import *
from proto_L2 import AMG2
nx=int(sys.argv[1]); mu=float(sys.argv[2]); dt=float(sys.argv[3]) if len(sys.argv)>3 else 0.01
prob,m=lid_problem(nx,mu,dt); n=prob.n
xk=np.zeros(3*n); un=np.zeros(2*n)
xk,its,reason=O.newton_solve(prob,xk,un,rtol=1e-6)
un=xk[:2*n].copy()
A=O.assemble_J(prob,xk[:2*n],xk[2*n:],un).tocsr(); b=O.assemble_F(prob,xk,un)
print('nu dt/h^2', mu/prob.rho*dt*nx*nx, 'N',3*n)
A00=A[:2*n,:2*n].tocsr(); A01=A[:2*n,2*n:].tocsr(); A10=A[2*n:,:2*n].tocsr(); A11=A[2*n:,2*n:].tocsr()
L,ml=laplace_mass(prob)
marker,g,mult=O.bc_arrays(prob)
unode=marker[:2*n:2]
keep=sp.diags((~unode).astype(float))
Lu=(keep@L@keep+sp.diags(unode.astype(float)*L.diagonal())).tocsr()
Lr=(L+1e-8*sp.diags(ml)).tocsr()
for sa in (True,):
    amgA=AMG2(A00,Lu,2,sa=sa,smoother='cheb',cheb_deg=int(sys.argv[4]) if len(sys.argv)>4 else 2)
    amgL=AMG2(Lr,L,1,sa=sa,smoother='cheb',cheb_deg=int(sys.argv[4]) if len(sys.argv)>4 else 2)
    rb=np.random.default_rng(1).standard_normal(2*n)
    x,its,res=fgmres(A00,rb,lambda r: amgA.cycle(r),rtol=1e-6,maxit=200); print('  A00 fgmres+V its',its,res)
    rb=np.random.default_rng(1).standard_normal(n); rb-=rb.mean()
    x,its,res=fgmres(Lr,rb,lambda r: amgL.cycle(r),rtol=1e-6,maxit=200); print('  L fgmres+V its',its,res)
    def proj(v): return v-v.mean()
    for nVu,nVp in ((1,1),(1,2),(2,2),(1,3),(2,4)):
        def ncyc(amg,Aop,v,k):
            z=amg.cycle(v)
            for _ in range(k-1): z=z+amg.cycle(v-Aop@z)
            return z
        def pc(r):
            ru=r[:2*n]; rp=proj(r[2*n:])
            zp=proj(mu*rp/ml+2*(prob.rho/dt)*ncyc(amgL,Lr,rp,nVp))
            zu=ncyc(amgA,A00,ru-A01@zp,nVu)
            return np.concatenate([zu,zp])
        x,its,res=fgmres(A,b,pc,rtol=1e-5,maxit=150)
        print(f'  outer SA={sa} nVu={nVu} nVp={nVp}: its {its} res {res:.2e}')
