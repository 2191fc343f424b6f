import os, sys, time; sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import numpy as np, scipy.sparse as sp, scipy.sparse.linalg as spla
from proto_pc import *
nx=int(sys.argv[1]); mu=float(sys.argv[2]); dt=float(sys.argv[3]) if len(sys.argv)>3 else 0.01
prob,m=lid_problem(nx,mu,dt); n=prob.n
xk=np.zeros(3*n); un=np.zeros(2*n)
xk,its,reason=O.newton_solve(prob,xk,un,rtol=1e-6)
un=xk[:2*n].copy()
A=O.assemble_J(prob,xk[:2*n],xk[2*n:],un).tocsr(); b=O.assemble_F(prob,xk,un)
print('nu dt/h^2', mu/prob.rho*dt*nx*nx, 'N',3*n)
A00=A[:2*n,:2*n].tocsc(); A01=A[:2*n,2*n:].tocsr(); A10=A[2*n:,:2*n].tocsr(); A11=A[2*n:,2*n:].tocsr()
L,ml=laplace_mass(prob)
lu00=spla.splu(A00)
Lr=(L+1e-10*sp.diags(ml)).tocsc(); luL=spla.splu(Lr)
Sp=(A11-A10@sp.diags(1/A00.diagonal())@A01).tocsc(); 
e=np.ones(n)/np.sqrt(n)
luSp=spla.splu((Sp+1e-10*sp.diags(ml)).tocsc())
def run(name,Sinv,fact='upper'):
    def pc(r):
        ru=r[:2*n]; rp=r[2*n:]
        if fact=='upper':
            zp=Sinv(rp); zu=lu00.solve(ru-A01@zp)
        elif fact=='diag':
            zp=Sinv(rp); zu=lu00.solve(ru)
        else:
            zu=lu00.solve(ru); zp=Sinv(rp-A10@zu); zu=zu-lu00.solve(A01@zp)
        return np.concatenate([zu,zp])
    x,its,res=fgmres(A,b,pc,rtol=1e-5,maxit=150)
    print(f'  {name} {fact}: its {its} res {res:.2e}')
def proj(v): return v-v.mean()
cc=lambda v: proj(mu*proj(v)/ml + 2*(prob.rho/dt)*luL.solve(proj(v)))
cc1=lambda v: proj(mu*proj(v)/ml + 1*(prob.rho/dt)*luL.solve(proj(v)))
selfp=lambda v: proj(luSp.solve(proj(v)))
for fact in ('upper','full'):
    run('CC(2rho/dt)',cc,fact); run('CC(rho/dt)',cc1,fact); run('SELFP',selfp,fact)
if n<3000:
    S=A11.toarray()-A10.toarray()@np.linalg.solve(A00.toarray(),A01.toarray())
    Si=np.linalg.pinv(S)
    run('exactS',lambda v: Si@v,'upper'); run('exactS',lambda v: Si@v,'full')
