import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from fugue_b200 import kernels as K
dev = torch.device("cuda", 0)
g = torch.Generator(device=dev).manual_seed(0)
n, nk = 125_000_000, 10_000_000
keys = torch.randint(0, nk, (n,), dtype=torch.int64, device=dev, generator=g) * 0x9E3779B97F4A7C15 % (1 << 62)
v = torch.randn(n, dtype=torch.float64, device=dev, generator=g).view(torch.int64)
for _ in range(2):
    K.groupby_u64(keys, None, [v, None], [None, None], [K.AGG_SUM_F64, K.AGG_COUNT])
torch.cuda.synchronize()
del keys, v
n = 62_500_000
lk = torch.randint(0, n, (n,), dtype=torch.int64, device=dev, generator=g)
rk = torch.randperm(n, dtype=torch.int64, device=dev, generator=g)
lv = torch.randn(n, dtype=torch.float64, device=dev, generator=g)
rv = torch.randn(n, dtype=torch.float64, device=dev, generator=g)
from fugue_b200 import api as fa
from fugue_b200.dataframe import B200DataFrame
from fugue_b200.table import B200Table
e = fa.make_execution_engine("b200")
L = B200DataFrame(B200Table("key:long,lv:double", [lk, lv]))
R = B200DataFrame(B200Table("key:long,rv:double", [rk, rv]))
for _ in range(2):
    e.join(L, R, "inner", ["key"])
torch.cuda.synchronize()
