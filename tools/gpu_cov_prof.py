"""k_cov_gemm2 launches at C = 16384, L = 1024, nsplit = 2 for ncu."""
import sys
import torch
sys.path.insert(0, ".")
from mmseq_b200 import capi
dev = torch.device("cuda:0")
L, C, nsplit = 1024, int(sys.argv[1]) if len(sys.argv) > 1 else 16384, int(sys.argv[2]) if len(sys.argv) > 2 else 2
g = torch.Generator(device=dev); g.manual_seed(1)
Md = torch.exp(torch.randn((C, L), dtype=torch.float64, device=dev, generator=g))
Rd = torch.empty((C, C), dtype=torch.float64, device=dev)
ws = torch.empty(capi.trace_cov_workspace_bytes(L, C, nsplit), dtype=torch.uint8, device=dev)
st = torch.cuda.current_stream()
for _ in range(3):
    capi.trace_cov_dev(Md.data_ptr(), L, C, nsplit, Rd.data_ptr(), ws.data_ptr(), st.cuda_stream)
torch.cuda.synchronize()
