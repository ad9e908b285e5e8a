import torch, json
from torch.profiler import profile, ProfilerActivity
from sparsearray_b200.device import DeviceSVT
x = DeviceSVT.generate_poisson(33538, 1000000, 0.07, seed=2, na_rate=1e-6)
y = DeviceSVT.generate_poisson(33538, 1000000, 0.07, seed=3, na_rate=1e-6)
r = x.ewise_svt("+", y); del r
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(3):
        r = x.ewise_svt("+", y); del r
    torch.cuda.synchronize()
out = {}
for e in prof.key_averages():
    if e.device_type.name == "CUDA" or "ewise2" in e.key:
        t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
        out[e.key[:90]] = round(t / 1e3 / max(e.count, 1), 3)
print(json.dumps(out))
