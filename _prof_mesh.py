import sys, numpy as np, torch
sys.path.insert(0, ".")
from dynamicfusion_b200 import capi, kinfu as kf, synth
lib = capi.load()
p = kf.KinFuParams.default_params_dynamicfusion(); kf.KinFuParams.set_volume(p, 512, 1.0); p.max_nodes = 2048; p.cloud_capacity = 4_000_000
k = kf.KinFu(p)
for t in range(40):
    d = torch.from_numpy(synth.umbrella_depth(t, seed=0).view(np.int16).copy()).cuda()
    lib.df_kinfu_process_device(k.h, d.data_ptr(), 1280)
k.info(); torch.cuda.synchronize()
cap = 4_000_000
v = torch.empty((cap, 4), device="cuda"); n = torch.empty_like(v); keys = torch.empty(cap, dtype=torch.int32, device="cuda")
tr = torch.empty((2 * cap, 3), dtype=torch.int32, device="cuda"); import ctypes as C; c = (C.c_int * 2)()
for _ in range(3): lib.df_kinfu_extract_mesh(k.h, 0, v.data_ptr(), n.data_ptr(), keys.data_ptr(), cap, tr.data_ptr(), 2 * cap, c)
from torch.profiler import profile, ProfilerActivity
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(10): lib.df_kinfu_extract_mesh(k.h, 0, v.data_ptr(), n.data_ptr(), keys.data_ptr(), cap, tr.data_ptr(), 2 * cap, c)
    torch.cuda.synchronize()
print(list(c))
print(prof.key_averages().table(sort_by="cuda_time_total", row_limit=15, max_name_column_width=70))
