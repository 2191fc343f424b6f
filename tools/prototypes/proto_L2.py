import os, sys, time; sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import numpy as np, scipy.sparse as sp
from proto_pc import *

class AMG2(AMG):
    """adds: smoothed aggregation prolongator + K-cycle"""
    def __init__(self, A, graph, bs, sa=False, kcycle=0, **kw):
        self.sa=sa; self.kc=kcycle
        self.levels=[]; self.bs=bs
        self.nsm=kw.get('nsm',1); self.over=kw.get('over',1.0); self.smoother=kw.get('smoother','cheb'); self.omega=kw.get('omega',0.7); self.cheb_deg=kw.get('cheb_deg',2)
        theta=kw.get('theta',0.0); max_coarse=kw.get('max_coarse',200)
        G=graph.tocsr()
        while True:
            n=G.shape[0]; lev={'A':A.tocsr()}; lev['Dinv']=1.0/A.diagonal()
            DA=sp.diags(lev['Dinv'])@lev['A']; v=np.random.default_rng(0).standard_normal(A.shape[0])
            for _ in range(15):
                v=DA@v; lam=np.linalg.norm(v); v/=lam
            lev['lmax']=1.1*lam
            self.levels.append(lev)
            if n<=max_coarse: break
            S=strength(G,theta); agg,na=aggregate(S)
            Pn=sp.csr_matrix((np.ones(n),(np.arange(n),agg)),shape=(n,na))
            if sa:
                Dg=1.0/G.diagonal(); 
                v=np.random.default_rng(0).standard_normal(n)
                for _ in range(15):
                    v=Dg*(G@v); lam=np.linalg.norm(v); v/=lam
                Pn=(Pn - (4.0/3.0/lam)*sp.diags(Dg)@G@Pn).tocsr()
            P=sp.kron(Pn,sp.eye(bs)).tocsr() if bs>1 else Pn
            lev['P']=P; lev['R']=P.T.tocsr()
            A=(P.T@A@P).tocsr(); G=(Pn.T@G@Pn).tocsr()
        self.coarse=np.linalg.pinv(self.levels[-1]['A'].toarray())
        print('  levels',[l['A'].shape[0] for l in self.levels],'opc',sum(l['A'].nnz for l in self.levels)/self.levels[0]['A'].nnz)
    def cycle(self,b,l=0):
        lev=self.levels[l]
        if l==len(self.levels)-1: return self.coarse@b
        x=self.smooth(lev,np.zeros_like(b),b)
        r=b-lev['A']@x; rc=lev['R']@r
        if self.kc and l+1<len(self.levels)-1 and l<self.kc:
            Ac=self.levels[l+1]['A']
            # 2 its of GCR preconditioned by cycle(l+1)
            ec=np.zeros_like(rc); rr=rc.copy(); Ps=[];APs=[]
            for it in range(2):
                z=self.cycle(rr,l+1); az=Ac@z
                for p_,ap_ in zip(Ps,APs):
                    beta=(ap_@az)/(ap_@ap_); z=z-beta*p_; az=az-beta*ap_
                alpha=(az@rr)/(az@az); ec+=alpha*z; rr-=alpha*az; Ps.append(z);APs.append(az)
        else:
            ec=self.over*self.cycle(rc,l+1)
        x=x+lev['P']@ec
        return self.smooth(lev,x,b)
    def vcycle(self,b,l=0,x=None): return self.cycle(b,l)

if __name__=='__main__':
  for nx in (128,256,512):
    m=M.create_unit_square(None,nx,nx)
    class P_: pass
    prob=P_(); prob.x=m.geometry.x[:,:2]; prob.cells=m.geometry.dofmap; prob.n=prob.x.shape[0]
    L,ml=laplace_mass(prob); n=prob.n
    Lr=(L+1e-8*sp.diags(ml)).tocsr()
    rb=np.random.default_rng(1).standard_normal(n); rb-=rb.mean()
    for name,kw in (('plainV',dict(over=1.8)),('K-cycle',dict(kcycle=10)),('K2',dict(kcycle=2,over=1.8)),('SA',dict(sa=True))):
        amg=AMG2(Lr,L,1,smoother='cheb',cheb_deg=3,**kw)
        x,its,res=fgmres(Lr,rb,lambda r: amg.cycle(r),rtol=1e-6,maxit=200)
        print(f'nx {nx} {name}: its(1e-6) {its}')
