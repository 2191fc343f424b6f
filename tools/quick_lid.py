import os, sys, time; sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from cfd_hemodynamic_b200.src.scenarios.lid_driven2D import LidDriven2DSimulation
nx=int(sys.argv[1]); mu=float(sys.argv[2]); steps=int(sys.argv[3])
kw={}
for a in sys.argv[4:]:
    k,v=a.split('='); kw[k]=eval(v)
t0=time.time()
sc=LidDriven2DSimulation("stabilized_schur",0.01,1.0,rho=1,mu=mu,nx=nx,**kw)
s=sc.solver
torch.cuda.synchronize(); print('setup s',time.time()-t0,'levels',[[l['P'].shape for l in lv] for lv in s.linear.levels])
for i in range(steps):
    l0=s.hemo.launches
    torch.cuda.synchronize(); t1=time.time()
    s.step_device()
    torch.cuda.synchronize(); dt=time.time()-t1
    print(f'step {i}: {dt*1e3:.1f} ms newton {s.its_snes} ksp {s.its_ksp} reason {s.reason} launches {s.hemo.launches-l0}')
