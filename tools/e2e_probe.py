import os, sys, time, torch, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from openwebrx_b200 import ChannelBank
from openwebrx_b200.synth import BANDPASS, carrier_plan
FS=10_000_000; BLOCK=1<<24
cars=carrier_plan(64,FS,seed=20260101)
h=torch.randn(BLOCK,2).mul_(1e-3).pin_memory()
d=torch.empty(BLOCK,2,device='cuda')
torch.cuda.synchronize()
for _ in range(3):
    t0=time.perf_counter(); d.copy_(h,non_blocking=True); torch.cuda.synchronize(); t=time.perf_counter()-t0
print("H2D 134MB pinned: %.2f ms (%.1f GB/s)"%(t*1e3, BLOCK*8/t/1e9))
bank=ChannelBank(FS)
ch=[bank.add_channel(12000,demod=c["kind"],offset=c["offset"],bandpass=BANDPASS[c["kind"]]) for c in cars]
hp=h.data_ptr()
buf=np.empty((len(ch),1<<15),np.float32)
def step():
    bank.feed_ptr(hp,BLOCK)
    return sum(bank.read_audio_all(ch,buf))
for i in range(3): step()
s0=bank.stats()
t0=time.perf_counter()
for i in range(10): step()
t=(time.perf_counter()-t0)/10
s1=bank.stats()
print("feed+read wall %.2f ms, device ev0->ev1 %.2f ms"%(t*1e3,(s1['device_ms']-s0['device_ms'])/10))
t0=time.perf_counter(); n=sum(len(c.read_audio()) for c in ch); print("read_audio all: %.2f ms, %d samples"%((time.perf_counter()-t0)*1e3,n))
