import os, time, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tests import golden_io
from turbo_b200 import engine, abi
pb,_=golden_io.load('trains15')
for i in range(4):
    t0=time.perf_counter(); s=engine.Solver(pb, cutnodes=2000); t1=time.perf_counter()
    r=s.solve(); t2=time.perf_counter(); s.close(); t3=time.perf_counter()
    print(f"create {1e3*(t1-t0):.1f} ms solve {1e3*(t2-t1):.1f} ms (kernel {r['stats']['kernel_ms']:.1f}) destroy {1e3*(t3-t2):.1f} ms")
