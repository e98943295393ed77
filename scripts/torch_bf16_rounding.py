"""How torch's CUDA ops round the bf16 intermediates of sampling.py (division by a Python float, softmax, cumsum, compare),
against correctly rounded restatements.  Needs a CUDA device; prints one block (profiles/r03b_torch_bf16_rounding.log)."""
import torch
import torch.nn.functional as F

dev = "cuda"
print(torch.__version__, torch.cuda.get_device_name(0))
bits = torch.arange(0, 65536, dtype=torch.int32).to(torch.int16)
allbf = bits.view(torch.bfloat16)
fin = torch.isfinite(allbf.float())
allbf = allbf[fin]
print("finite bf16 values", allbf.numel())
for T in [0.9, 0.05, 3.0, 0.8, 0.7, 1.1, 1.3, 0.6, 1.5]:
    cu = (allbf.to(dev) / T).cpu()
    x32 = allbf.float()
    t32 = torch.tensor(T, dtype=torch.float32)
    div = (x32 / t32).to(torch.bfloat16)
    rcp = (x32 * (1.0 / t32)).to(torch.bfloat16)
    cpu = allbf / T
    f = lambda a, b: int((a.float() != b.float()).sum())
    print(f"T={T}: cuda!=div {f(cu, div)}  cuda!=rcp {f(cu, rcp)}  cpu!=div {f(cpu, div)}  cpu!=cuda {f(cpu, cu)}")

g = torch.Generator().manual_seed(0)
n_sm = n_cs_f = n_cs_seq = n_cs_cpu = tot = 0
set_diff = {}
for trial in range(200):
    V = [3072, 2048, 257][trial % 3]
    lg = (3.0 * torch.randn(1, V, generator=g)).to(torch.bfloat16)
    x = (lg.to(dev) / 0.9)
    kth = torch.topk(x, 50 if trial % 2 else V).values[..., -1:]
    x = torch.where(x < kth, torch.full_like(x, float("-inf")), x)
    srt, idx = torch.sort(x, descending=True, stable=True)
    sm = F.softmax(srt, dim=-1)
    sm_ref = F.softmax(srt.float(), dim=-1).to(torch.bfloat16)
    n_sm += int((sm != sm_ref).sum())
    cs = torch.cumsum(sm, dim=-1).cpu()
    smc = sm.cpu()
    cs_f = torch.cumsum(smc.double(), dim=-1).to(torch.float32).to(torch.bfloat16)
    acc = torch.zeros((), dtype=torch.bfloat16)
    seq = torch.empty_like(smc)
    for j in range(V):
        acc = (acc + smc[0, j])
        seq[0, j] = acc
    cs_cpu = torch.cumsum(smc, dim=-1)
    n_cs_f += int((cs != cs_f).sum()); n_cs_seq += int((cs != seq).sum()); n_cs_cpu += int((cs != cs_cpu).sum()); tot += V
    for p in (0.8, 0.95, 0.5):
        a = int((cs > p).logical_not().sum()); b = int((cs_f > p).logical_not().sum()); c = int((seq > p).logical_not().sum())
        set_diff.setdefault(p, [0, 0, 0])
        set_diff[p][0] += a != b; set_diff[p][1] += a != c; set_diff[p][2] += 1
print(f"softmax bf16 cuda != round(fp32 softmax): {n_sm} of {tot}")
print(f"cumsum bf16 cuda != round(exact prefix): {n_cs_f}; != sequential bf16: {n_cs_seq}; != cpu cumsum: {n_cs_cpu} of {tot}")
print("top-p kept count differs (cuda vs exact-rounded, cuda vs sequential, rows):", set_diff)
x = torch.tensor([[0.8008, 0.80078125, 0.8, 0.79]], dtype=torch.bfloat16, device=dev)
print("bf16 > 0.8 on cuda:", (x > 0.8).tolist(), x.tolist())
z = torch.tensor([0.0, -0.0, 1.0, -0.0, 0.0, -1.0, 0.0], device=dev)
s, i = torch.sort(z, descending=True, stable=True)
print("stable sort of +-0 on cuda:", i.tolist(), s.tolist())
print("topk with ties:", torch.topk(z, 3).values.tolist())
zb = z.to(torch.bfloat16)
s, i = torch.sort(zb, descending=True, stable=True)
print("stable sort bf16 +-0 on cuda:", i.tolist())
