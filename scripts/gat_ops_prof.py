import os, sys, argparse
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch, bench, dgg_b200, model as models
import torch.nn.functional as F
from torch.profiler import profile, ProfilerActivity
shape = bench.PUBMED; dev = torch.device("cuda"); n = shape["n"]
hs = bench.make_set(shape, 0)
ii = hs["idx"].to(dev); nl = ii[:, ii[0] != ii[1]].contiguous()
adj = torch.sparse_coo_tensor(nl, torch.ones(nl.shape[1], device=dev), (n, n)).coalesce()
x = hs["x"].to(dev)
torch.manual_seed(0)
net = models.GAT_DGG_00(nfeat=shape["f"], nlayers=2, nhidden=shape["h"], nclass=3, args=argparse.Namespace(extra_edge_dim=0, dgg_adj_input="input_adj")).to(dev)
opt = torch.optim.Adam(net.parameters(), lr=0.005, weight_decay=5e-4, fused=True)
labels = torch.randint(0, 3, (n,), device=dev); ti = torch.arange(60, device=dev)
def body():
    net.train(); opt.zero_grad(set_to_none=True)
    logp, _, _ = net(x, adj, edge_index=nl)
    loss = F.nll_loss(logp[ti], labels[ti]); loss.backward(); opt.step(); return loss
for i in range(5): body()
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA], record_shapes=True) as prof:
    for i in range(2): body()
    torch.cuda.synchronize()
print(prof.key_averages(group_by_input_shape=True).table(sort_by="cuda_time_total", row_limit=25, max_name_column_width=40, max_shapes_column_width=70))
