import os, sys; sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cvsteer_b200.batch import ffma_peak
for f,n in ((0,'ffma imm'),(1,'ffma reg'),(3,'ffma2 (lane-FMAs)'),(4,'ffma2 + alu 1:1 (lane-FMAs)'),(5,'ffma + alu 1:1')):
    v,ms=ffma_peak(f,20000); print(f'{n:32s} {v/1e12:7.2f} T/s  {ms:.2f} ms')
