import os, sys, time; sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import numpy as np, scipy.sparse as sp, scipy.sparse.linalg as spla
from proto_pc import *
nx=int(sys.argv[1]); mu=float(sys.argv[2]); dt=float(sys.argv[3]) if len(sys.argv)>3 else 0.01
prob,m=lid_problem(nx,mu,dt); n=prob.n
xk=np.zeros(3*n); un=np.zeros(2*n)
t0=time.time()
xk,its,reason=O.newton_solve(prob,xk,un,rtol=1e-6)
un=xk[:2*n].copy(); print('newton',its,reason,time.time()-t0)
A=O.assemble_J(prob,xk[:2*n],xk[2*n:],un).tocsr(); b=O.assemble_F(prob,xk,un)
print('nu dt/h^2', mu/prob.rho*dt*nx*nx, 'N',3*n)
A00=A[:2*n,:2*n].tocsr(); A01=A[:2*n,2*n:].tocsr(); A10=A[2*n:,:2*n].tocsr(); A11=A[2*n:,2*n:].tocsr()
L,ml=laplace_mass(prob)
marker,g,mult=O.bc_arrays(prob)
# nodal graph for aggregation: Laplacian
for smoother,kw in (('cheb',dict(cheb_deg=3)),):
  for over in (1.5,):
    print(f'== smoother {smoother} {kw} over {over}')
    amgA=AMG(A00,L,2,theta=0.0,smoother=smoother,over=over,**kw)
    Lr=L+1e-8*sp.diags(ml)   # regularise Neumann
    amgL=AMG(Lr.tocsr(),L,1,theta=0.0,smoother=smoother,over=over,**kw)
    # standalone quality: A00 solve convergence with V-cycle-preconditioned GMRES
    rb=np.random.default_rng(1).standard_normal(2*n)
    x,its,res=fgmres(A00,rb,lambda r: amgA.vcycle(r),rtol=1e-6,maxit=200); print('  A00 fgmres+V its',its,res)
    rb=np.random.default_rng(1).standard_normal(n); rb-=rb.mean()
    x,its,res=fgmres(Lr,rb,lambda r: amgL.vcycle(r),rtol=1e-6,maxit=200); print('  L fgmres+V its',its,res)
    for nV in (1,2):
      for fact in ('upper',):
        def pc(r):
            ru=r[:2*n]; rp=r[2*n:]
            def A00inv(v):
                z=amgA.vcycle(v)
                for _ in range(nV-1):
                    z=z+amgA.vcycle(v-A00@z)
                return z
            def Sinv(v):
                v=v-v.mean()
                z=(mu)*v/ml + 2*(prob.rho/dt)*amgL.vcycle(v)
                return z-z.mean()
            if fact=='upper':
                zp=Sinv(rp); zu=A00inv(ru-A01@zp)
            else:
                zu=A00inv(ru); zp=Sinv(rp-A10@zu); zu=zu-A00inv(A01@zp)
            return np.concatenate([zu,zp])
        x,its,res=fgmres(A,b,pc,rtol=1e-5,maxit=150)
        print(f'  outer nV={nV} {fact}: its {its} res {res:.2e}')
