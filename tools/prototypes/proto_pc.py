"""Prototype (scipy) of the block preconditioner to pick the algorithm before
writing CUDA.  Not product code."""
import os, sys, time; sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import numpy as np, scipy.sparse as sp, scipy.sparse.linalg as spla
from cfd_hemodynamic_b200.fem import mesh as M, quadrature as Q
from oracle import ns_oracle as O

def lid_problem(nx, mu, dt=0.01, rho=1.0, deg=4):
    m = M.create_unit_square(None, nx, nx)
    x = m.geometry.x[:, :2].copy(); cells = m.geometry.dofmap
    rule = Q.triangle_gauss_jacobi(deg)
    rules = {k: rule for k in ('Fu','Fp','uu','up','pu','pp')}
    prob = O.Problem(x=x, cells=cells, h=O.cell_diameter(x,cells), dt=dt, rho=rho, mu=mu, f=np.zeros(2), rules=rules, facet_rule=Q.interval_gauss(2))
    n=prob.n
    ext = M.exterior_facet_indices(m.topology)
    prob.facet_sets=[O.FacetSet(pairs=m.topology.facet_cell_pairs(ext), a_p=1.0, a_g=1.0)]
    walls = np.nonzero(np.isclose(x[:,0],0)|np.isclose(x[:,0],1)|np.isclose(x[:,1],0))[0]
    lidf = M.locate_entities_boundary(m,1,lambda X: np.isclose(X[1],1.0)&(X[0]>1e-10)&(X[0]<1-1e-10))
    lid = np.unique(m.topology.facet_vertices[lidf])
    g0=np.zeros(2*n); g1=np.zeros(2*n); g1[0::2]=1.0
    ud=lambda nodes: (2*nodes[:,None]+np.arange(2)[None]).ravel()
    prob.bcs=[('u',ud(walls),g0),('u',ud(lid),g1)]
    return prob, m

def aggregate(S):
    """greedy aggregation on strength graph S (csr, symmetric pattern, no diag)."""
    n = S.shape[0]; ip, ix = S.indptr, S.indices
    agg = -np.ones(n, dtype=np.int64); na = 0
    for i in range(n):
        if agg[i] >= 0: continue
        nb = ix[ip[i]:ip[i+1]]
        if np.all(agg[nb] < 0):
            agg[i] = na; agg[nb] = na; na += 1
    for i in range(n):
        if agg[i] >= 0: continue
        nb = ix[ip[i]:ip[i+1]]
        a = agg[nb]; a = a[a >= 0]
        if len(a): agg[i] = -2 - a[0]   # tentative
    t = agg <= -2
    agg[t] = -2 - agg[t]
    for i in range(n):
        if agg[i] == -1:
            agg[i] = na; nb = ix[ip[i]:ip[i+1]]
            for j in nb:
                if agg[j] == -1: agg[j] = na
            na += 1
    return agg, na

def strength(A, theta):
    A = A.tocsr(); d = np.abs(A.diagonal())
    C = A.tocoo()
    mask = (C.row != C.col) & (np.abs(C.data) >= theta*np.sqrt(d[C.row]*d[C.col]))
    return sp.csr_matrix((np.ones(mask.sum()), (C.row[mask], C.col[mask])), shape=A.shape)

class AMG:
    def __init__(self, A, graph, bs, theta=0.25, max_coarse=200, smoother='jacobi', omega=0.7, nsm=1, over=1.0, cheb_deg=2):
        """A: (bs*n) matrix with node-interleaved dofs; graph: scalar nodal matrix for strength."""
        self.levels = []; self.bs = bs; self.nsm=nsm; self.over=over; self.smoother=smoother; self.omega=omega; self.cheb_deg=cheb_deg
        G = graph.tocsr()
        while True:
            n = G.shape[0]
            lev = {'A': A.tocsr()}
            lev['Dinv'] = 1.0/A.diagonal()
            # l1-ish / spectral radius estimate for Chebyshev
            if smoother=='cheb':
                DA = sp.diags(lev['Dinv'])@lev['A']
                v = np.random.default_rng(0).standard_normal(A.shape[0])
                for _ in range(15):
                    v = DA@v; lam = np.linalg.norm(v); v/=lam
                lev['lmax']=1.1*lam
            self.levels.append(lev)
            if n <= max_coarse: break
            S = strength(G, theta)
            agg, na = aggregate(S)
            Pn = sp.csr_matrix((np.ones(n), (np.arange(n), agg)), shape=(n, na))
            P = sp.kron(Pn, sp.eye(bs)).tocsr() if bs > 1 else Pn
            lev['P'] = P; lev['R'] = P.T.tocsr()
            A = (P.T @ A @ P).tocsr(); G = (Pn.T @ G @ Pn).tocsr()
        Ac = self.levels[-1]['A'].toarray()
        self.coarse = np.linalg.pinv(Ac)
        print('  levels', [l['A'].shape[0] for l in self.levels], 'opc', sum(l['A'].nnz for l in self.levels)/self.levels[0]['A'].nnz)
    def smooth(self, lev, x, b):
        A = lev['A']; Dinv = lev['Dinv']
        if self.smoother=='jacobi':
            for _ in range(self.nsm):
                x = x + self.omega*Dinv*(b - A@x)
            return x
        else:  # chebyshev on D^-1 A with [lmax/a, lmax]
            lmax = lev['lmax']; lmin = lmax/4.0
            theta=(lmax+lmin)/2; delta=(lmax-lmin)/2
            r = Dinv*(b - A@x); sigma=theta/delta; rho=1/sigma
            d = r/theta
            for k in range(self.cheb_deg):
                x = x + d
                if k==self.cheb_deg-1: break
                r = r - Dinv*(A@d)
                rho_new = 1/(2*sigma-rho)
                d = rho_new*rho*d + 2*rho_new/delta*r
                rho=rho_new
            return x
    def vcycle(self, b, l=0, x=None):
        lev = self.levels[l]
        if l == len(self.levels)-1:
            return self.coarse @ b
        x = np.zeros_like(b)
        x = self.smooth(lev, x, b)
        r = b - lev['A']@x
        ec = self.vcycle(lev['R']@r, l+1)
        x = x + self.over*(lev['P']@ec)
        x = self.smooth(lev, x, b)
        return x

def fgmres(A, b, Minv, rtol=1e-5, restart=60, maxit=300, monitor=False):
    n=len(b); x=np.zeros(n); r=b.copy(); beta=np.linalg.norm(r); b0=beta; its=0
    while its<maxit:
        V=[r/beta]; Z=[]; H=np.zeros((restart+1,restart)); g=np.zeros(restart+1); g[0]=beta
        cs=[];sn=[]
        for j in range(restart):
            z=Minv(V[j]); Z.append(z); w=A@z
            for i in range(j+1):
                H[i,j]=V[i]@w
            for i in range(j+1): w=w-H[i,j]*V[i]
            H[j+1,j]=np.linalg.norm(w); V.append(w/H[j+1,j])
            for i in range(j):
                t=cs[i]*H[i,j]+sn[i]*H[i+1,j]; H[i+1,j]=-sn[i]*H[i,j]+cs[i]*H[i+1,j]; H[i,j]=t
            d=np.hypot(H[j,j],H[j+1,j]); cs.append(H[j,j]/d); sn.append(H[j+1,j]/d)
            H[j,j]=d; H[j+1,j]=0; g[j+1]=-sn[j]*g[j]; g[j]=cs[j]*g[j]
            its+=1
            if monitor: print('   ',its,abs(g[j+1])/b0)
            if abs(g[j+1])<=rtol*b0 or its>=maxit:
                j+=1;break
        else: j=restart
        y=np.linalg.solve(np.triu(H[:j,:j]),g[:j])
        for i in range(j): x+=y[i]*Z[i]
        r=b-A@x; beta=np.linalg.norm(r)
        if beta<=rtol*b0: break
    return x,its,beta/b0

def laplace_mass(prob):
    det,dphi=O.cell_geometry(prob.x,prob.cells)
    area=det/2
    Ke=area[:,None,None]*np.einsum('eai,ebi->eab',dphi,dphi)
    c=prob.cells
    rows=np.repeat(c,3,axis=1).ravel(); cols=np.tile(c,(1,3)).ravel()
    L=sp.coo_matrix((Ke.ravel(),(rows,cols)),shape=(prob.n,prob.n)).tocsr()
    ml=np.zeros(prob.n); np.add.at(ml,c.ravel(),np.repeat(area/3,3))
    return L,ml

if __name__=='__main__':
    nx=int(sys.argv[1]); mu=float(sys.argv[2]); dt=float(sys.argv[3]) if len(sys.argv)>3 else 0.01
    prob,m=lid_problem(nx,mu,dt)
    n=prob.n
    # state: run 1 newton step with splu to get a nontrivial velocity
    xk=np.zeros(3*n); un=np.zeros(2*n)
    t0=time.time()
    xk,its,reason=O.newton_solve(prob,xk,un,rtol=1e-6)
    un=xk[:2*n].copy(); print('newton',its,reason,time.time()-t0)
    A=O.assemble_J(prob,xk[:2*n],xk[2*n:],un); b=O.assemble_F(prob,xk,un)
    print('nu dt/h^2', mu/prob.rho*dt*nx*nx)
    np.save('/tmp/proto_b.npy', b); sp.save_npz('/tmp/proto_A.npz', A)
