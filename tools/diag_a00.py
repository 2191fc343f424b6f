import sys, os; sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import contextlib, numpy as np, torch, scipy.sparse as sp
from cfd_hemodynamic_b200.src.scenarios.stenosis_mesh_variable import StenosisMeshVariableSimulation as S
with contextlib.redirect_stdout(sys.stderr):
    sc = S("stabilized_schur_backflow", 1e-3, 1.0, grade="severe", v_max=100.0, res=float(sys.argv[1]))
s = sc.solver
for i in range(3): s.step_device()
h = s.hemo; n = s.n
h.assemble_jacobian(s.d_x, s.d_un, s.d_vals); s.linear.setup(s.d_vals)
rowptr, col = h.get_pattern()
A = sp.csr_matrix((s.d_vals.cpu().numpy(), col.cpu().numpy(), rowptr.cpu().numpy()), shape=(3*n, 3*n))
A00 = A[:2*n, :2*n].tocsr(); A11 = A[2*n:, 2*n:].tocsr(); A01 = A[:2*n, 2*n:].tocsr(); A10 = A[2*n:, :2*n].tocsr()
rng = np.random.default_rng(0)
b = rng.standard_normal(2*n); bd = torch.tensor(b, device=h.device); xd = torch.zeros_like(bd)
for k in (1, 2, 4, 8):
    h.amg_apply(0, bd, xd, k)
    print("A00 V-cycles", k, "rel res", np.linalg.norm(b - A00 @ xd.cpu().numpy()) / np.linalg.norm(b))
# smooth rhs
xs = s.mesh.geometry.x[:, :2]
bs = np.stack([np.sin(xs[:,0]/10)*np.cos(xs[:,1]), np.cos(xs[:,0]/7)], 1).ravel(); bs[np.abs(A00.diagonal()-1)<1e-14] = 0
bd = torch.tensor(bs, device=h.device)
for k in (1, 2, 4, 8):
    h.amg_apply(0, bd, xd, k)
    print("A00 smooth rhs V-cycles", k, "rel res", np.linalg.norm(bs - A00 @ xd.cpu().numpy()) / np.linalg.norm(bs))
d = A00.diagonal(); print("diag dominance: min |a_ii|/sum|a_ij| ", float((np.abs(d) / (np.abs(A00).sum(axis=1).A1 - np.abs(d) + 1e-300)).min()))
# magnitude of Schur pieces along a few random vectors
import scipy.sparse.linalg as spla
print("||A11|| est", spla.norm(A11, 'fro') / np.sqrt(n), " ||A10 D^-1 A01|| est", spla.norm(A10 @ sp.diags(1/d) @ A01, 'fro') / np.sqrt(n))
