import os,sys,time
sys.path.insert(0,os.path.join(os.path.dirname(os.path.abspath(__file__)),'..'))
import torch
from bioem_b200 import api
from bioem_b200.cases import build_case
cd=build_case('cfg2', n_particles=64)
hi,parts=api.inputs_for_case(cd)
eng=api.Engine(hi.cfg,0); eng.upload_all(hi,parts); eng.set_kernel_timing(True)
# time debug_projection-like front end: use run on tiny M so that the front end dominates? -> time run_front via stats
eng.reset(); eng.run(0,150); eng.synchronize(); eng.kernel_time()
t=time.time(); eng.reset(); eng.run(0,600); eng.synchronize(); dt=time.time()-t
ms,n=eng.kernel_time()
print(f"band_kb={os.environ.get('BIOEM_B200_BAND_KB','default')}: 600 orientations x 64 particles: total {dt*1e3:.1f} ms, likelihood kernels {ms:.1f} ms, front+rest {dt*1e3-ms:.1f} ms")
