"""Generate tests/golden/*.pt by RUNNING THE REFERENCE'S OWN FILES in the authoring container.

    PNA_REFERENCE=<reference checkout> PYTHONPATH=. python oracle/gen_golden.py [--round2 | --propagate]

/root/reference's PyG and DGL layers import torch_geometric / torch_scatter / dgl, none of which exist here; they are
imported over the minimal third-party restatements in oracle/shims/ (see its README).  The files under test --
models/pytorch_geometric/pna.py, aggregators.py, scalers.py, models/dgl/pna_layer.py, aggregators.py, scalers.py,
models/pytorch/pna/*.py, multitask_benchmark/datasets_generation/*.py -- are the reference's, unmodified.

Every fixture stores inputs, constructor arguments, the layer's state_dict and the reference outputs, so that
tests can (a) pin oracle/pna_oracle.py and (b) load the state_dict into the pna_b200 drop-in layers on the GPU.
TEST INFRASTRUCTURE ONLY.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("PNA_REFERENCE", "/root/reference")
sys.path[:0] = [os.path.join(HERE, "shims"), REF, os.path.join(REF, "multitask_benchmark")]
OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")

from models.pytorch_geometric.pna import PNAConv, PNAConvSimple  # noqa: E402
from models.dgl.pna_layer import PNALayer as DGLPNALayer, PNASimpleLayer as DGLPNASimpleLayer  # noqa: E402
from models.pytorch.pna.layer import PNALayer as DensePNALayer  # noqa: E402
from models.pytorch.pna import aggregators as dense_aggr, scalers as dense_scal  # noqa: E402
from datasets_generation.graph_generation import generate_graph, GraphType  # noqa: E402
from datasets_generation.graph_algorithms import map_reduce_neighbourhood  # noqa: E402
import dgl  # noqa: E402  (shim)

A4 = ["mean", "max", "min", "std"]            # realworld_benchmark/configs/*.json order
A4_EX = ["mean", "min", "max", "std"]         # models/pytorch_geometric/example.py:33 order
S3 = ["identity", "amplification", "attenuation"]


def deg_hist(dst, n):
    return torch.bincount(torch.bincount(dst, minlength=n))


def graph_random(n, e, seed, isolated=0.2):
    """random multigraph with duplicates, self loops and ~isolated fraction of nodes without in-edges"""
    g = torch.Generator().manual_seed(seed)
    live = max(1, int(n * (1 - isolated)))
    dst = torch.randint(0, live, (e,), generator=g)
    src = torch.randint(0, n, (e,), generator=g)
    src[: e // 20] = dst[: e // 20]                      # self loops
    src[e // 20: e // 10] = src[0]; dst[e // 20: e // 10] = dst[0]   # duplicated edge
    return torch.stack([src, dst])


def graph_hub(n, e, hub_deg, seed):
    ei = graph_random(n, e, seed)
    g = torch.Generator().manual_seed(seed + 1)
    hub_src = torch.randint(0, n, (hub_deg,), generator=g)
    hub = torch.stack([hub_src, torch.full((hub_deg,), n - 1)])
    perm = torch.randperm(e + hub_deg, generator=g)
    return torch.cat([ei, hub], 1)[:, perm]


def save(name, obj):
    path = os.path.join(OUT, name + ".pt")
    torch.save(obj, path)
    print(f"{name}: {os.path.getsize(path) / 1024:.0f} KiB")


def simple_case(name, n, e, f, seed, aggrs=A4, scalers=S3, hub=0, constant_rows=False, post_layers=1):
    torch.manual_seed(seed)
    ei = graph_hub(n, e, hub, seed) if hub else graph_random(n, e, seed)
    x = torch.randn(n, f)
    if constant_rows:   # ZINC-like: few distinct embedding rows -> zero-variance neighbourhoods (std adversarial)
        table = torch.randn(4, f)
        x = table[torch.randint(0, 4, (n,))]
    deg = deg_hist(ei[1], n)
    conv = PNAConvSimple(f, f, aggrs, scalers, deg, post_layers=post_layers)
    with torch.no_grad():
        agg = conv.propagate(ei, x=x, size=None)
        out = conv(x, ei)
    save(name, dict(kind="pyg_simple", x=x, edge_index=ei, deg=deg, aggregators=aggrs, scalers=scalers,
                    post_layers=post_layers, avg_deg=conv.avg_deg, state_dict=conv.state_dict(), aggregate=agg, out=out))


def conv_case(name, n, e, fin, fout, seed, towers=1, divide_input=False, pre_layers=1, post_layers=1, edge_dim=None):
    torch.manual_seed(seed)
    ei = graph_random(n, e, seed)
    x = torch.randn(n, fin)
    ea = torch.randn(e, edge_dim) if edge_dim else None
    deg = deg_hist(ei[1], n)
    conv = PNAConv(fin, fout, A4, S3, deg, edge_dim=edge_dim, towers=towers, pre_layers=pre_layers,
                   post_layers=post_layers, divide_input=divide_input)
    with torch.no_grad():
        xt = x.view(-1, towers, conv.F_in) if divide_input else x.view(-1, 1, conv.F_in).repeat(1, towers, 1)
        agg = conv.propagate(ei, x=xt, edge_attr=ea, size=None)
        out = conv(x, ei, ea)
    save(name, dict(kind="pyg_conv", x=x, edge_index=ei, edge_attr=ea, deg=deg, aggregators=A4, scalers=S3,
                    ctor=dict(in_channels=fin, out_channels=fout, edge_dim=edge_dim, towers=towers, pre_layers=pre_layers,
                              post_layers=post_layers, divide_input=divide_input),
                    avg_deg=conv.avg_deg, state_dict=conv.state_dict(), aggregate=agg, out=out))


def dgl_cases():
    torch.manual_seed(7)
    n, e, f = 90, 400, 20
    ei = graph_random(n, e, 7)
    h = torch.randn(n, f)
    indeg = torch.bincount(ei[1], minlength=n).float()
    avg_d = dict(lin=indeg.mean().item(), exp=torch.exp(indeg).mean().item(), log=torch.log(indeg + 1).mean().item())
    snorm = torch.full((n, 1), 1.0 / np.sqrt(n))
    aggr, scal = "mean max min std", "identity amplification attenuation"
    lay = DGLPNASimpleLayer(f, f, aggr, scal, avg_d, dropout=0.0, batch_norm=True, residual=True, posttrans_layers=1)
    lay.eval()
    g = dgl.DGLGraph(ei[0], ei[1], n)
    with torch.no_grad():
        g.ndata["h"] = h
        g.update_all(dgl.function.copy_u("h", "m"), lay.reduce_func)
        agg = g.ndata["h"].clone()
        out = lay(dgl.DGLGraph(ei[0], ei[1], n), h)
    save("dgl_simple", dict(kind="dgl_simple", h=h, edge_index=ei, avg_d=avg_d, aggregators=aggr, scalers=scal,
                            ctor=dict(in_dim=f, out_dim=f, dropout=0.0, batch_norm=True, residual=True, posttrans_layers=1),
                            state_dict=lay.state_dict(), aggregate=agg, out=out))
    for name, kw, ef in (("dgl_layer_t5", dict(towers=5, divide_input=True, edge_features=False, edge_dim=0), None),
                         ("dgl_layer_edge", dict(towers=5, divide_input=False, edge_features=True, edge_dim=6, pretrans_layers=2,
                                                 posttrans_layers=2), torch.randn(e, 6))):
        lay = DGLPNALayer(f, f, aggr, scal, avg_d, dropout=0.0, graph_norm=True, batch_norm=True, residual=True, **kw)
        lay.eval()
        with torch.no_grad():
            out = lay(dgl.DGLGraph(ei[0], ei[1], n), h, ef, snorm)
        save(name, dict(kind="dgl_layer", h=h, e=ef, snorm_n=snorm, edge_index=ei, avg_d=avg_d, aggregators=aggr,
                        scalers=scal, ctor=dict(in_dim=f, out_dim=f, dropout=0.0, graph_norm=True, batch_norm=True,
                                                residual=True, **kw), state_dict=lay.state_dict(), out=out))


def dense_and_numpy_cases():
    """K1 (dense reference aggregators/scalers), K2 (numpy label reducers) and the dense layer on a generated graph."""
    torch.manual_seed(11)
    adj_np, feat_np, gtype = generate_graph(24, GraphType.ERDOS_RENYI, seed=1234, degree=4)
    # make sure no node is isolated (the reference generator rejects those graphs, multitask_dataset.py:46-49)
    for i in range(adj_np.shape[0]):
        if adj_np[i].sum() == 0:
            j = (i + 1) % adj_np.shape[0]
            adj_np[i, j] = adj_np[j, i] = 1
    adj = torch.tensor(adj_np, dtype=torch.float32).unsqueeze(0)
    n, f = adj.shape[1], 8
    h = torch.rand(1, n, f)
    avg_d = dict(lin=adj.sum(-1).mean().item(), log=torch.log(adj.sum(-1) + 1).mean().item())
    # K1: X[b,i,j,:] = h_j for mean/std/sum (reduce over j); X[b,i,j,:] = h_i for max/min (reduce over dim -3)
    X_j = h.unsqueeze(1).repeat(1, n, 1, 1)
    X_i = h.unsqueeze(2).repeat(1, 1, n, 1)
    k1 = dict(mean=dense_aggr.aggregate_mean(X_j, adj), std=dense_aggr.aggregate_std(X_j, adj),
              sum=dense_aggr.aggregate_sum(X_j, adj), max=dense_aggr.aggregate_max(X_i, adj),
              min=dense_aggr.aggregate_min(X_i, adj))
    m = torch.cat([k1["mean"], k1["max"], k1["min"], k1["std"]], dim=2)
    k1_scaled = torch.cat([dense_scal.SCALERS[s](m, adj, avg_d=avg_d) for s in S3], dim=2)
    # K2: float64 numpy reducers over the 1-hop neighbourhood, population std, no eps
    k2 = {nm: np.stack([map_reduce_neighbourhood(adj_np, h[0, :, c].numpy().astype(np.float64), fn) for c in range(f)], 1)
          for nm, fn in (("mean", np.mean), ("max", np.max), ("min", np.min), ("std", np.std))}
    lay = DensePNALayer(f, f, A4, S3, avg_d, towers=2, self_loop=False, pretrans_layers=1, posttrans_layers=1,
                        divide_input=True)
    lay.eval()
    with torch.no_grad():
        out = lay(h, adj)
    # gradients of a fixed scalar loss through the reference dense layer (multitask training path)
    gw = torch.randn(out.shape, generator=torch.Generator().manual_seed(3))
    hg = h.clone().requires_grad_(True)
    lay.zero_grad()
    (lay(hg, adj) * gw).sum().backward()
    grads = dict(h=hg.grad.clone(), w=gw, params={k: v.grad.clone() for k, v in lay.named_parameters()})
    save("dense_k1_k2", dict(kind="dense", adj=adj, h=h, avg_d=avg_d, k1=k1, k1_scaled=k1_scaled, grads=grads,
                             k2={k: torch.tensor(v) for k, v in k2.items()}, graph_type=str(gtype),
                             ctor=dict(in_features=f, out_features=f, towers=2, self_loop=False, pretrans_layers=1,
                                       posttrans_layers=1, divide_input=True),
                             state_dict=lay.state_dict(), out=out))


def multitask_case():
    """config 1 in miniature: a reference-generated graph through PNAConv(16,16,towers=4,divide_input=True)."""
    adj_np, _, _ = generate_graph(60, GraphType.BARABASI_ALBERT, seed=1235, degree=3)
    dst, src = np.nonzero(adj_np)                       # adj[i, j] != 0  =>  edge j -> i
    ei = torch.tensor(np.stack([src, dst]), dtype=torch.long)
    torch.manual_seed(42)
    x = torch.rand(adj_np.shape[0], 16)
    deg = deg_hist(ei[1], x.size(0))
    conv = PNAConv(16, 16, A4, S3, deg, towers=4, divide_input=True)
    with torch.no_grad():
        out = conv(x, ei)
        agg = conv.propagate(ei, x=x.view(-1, 4, 4), edge_attr=None, size=None)
    save("pyg_conv_multitask", dict(kind="pyg_conv", x=x, edge_index=ei, edge_attr=None, deg=deg, aggregators=A4, scalers=S3,
                                    ctor=dict(in_channels=16, out_channels=16, edge_dim=None, towers=4, pre_layers=1,
                                              post_layers=1, divide_input=True),
                                    avg_deg=conv.avg_deg, state_dict=conv.state_dict(), aggregate=agg, out=out))


def round2_cases():
    """Fixtures added in round 2 (the earlier ones are not regenerated): the flavours' relu(var) and the dense layer with
    self_loop=True on a DIRECTED adjacency, where row and column degrees differ."""
    # DGL simple layer with "var" and ZINC-like identical neighbour rows: E[m^2] - E[m]^2 cancels to +-1 ulp noise, the
    # reference's torch.relu (models/dgl/aggregators.py:22-26) turns the negative ones into exact zeros
    torch.manual_seed(21)
    n, e, f = 80, 360, 12
    ei = graph_random(n, e, 21)
    table = torch.randn(3, f) * 3.0
    h = table[torch.randint(0, 3, (n,))]
    indeg = torch.bincount(ei[1], minlength=n).float()
    avg_d = dict(lin=indeg.mean().item(), exp=torch.exp(indeg).mean().item(), log=torch.log(indeg + 1).mean().item())
    aggr, scal = "mean max min std var", "identity amplification attenuation"
    lay = DGLPNASimpleLayer(f, f, aggr, scal, avg_d, dropout=0.0, batch_norm=True, residual=True, posttrans_layers=1)
    lay.eval()
    g = dgl.DGLGraph(ei[0], ei[1], n)
    with torch.no_grad():
        g.ndata["h"] = h
        g.update_all(dgl.function.copy_u("h", "m"), lay.reduce_func)
        agg = g.ndata["h"].clone()
        out = lay(dgl.DGLGraph(ei[0], ei[1], n), h)
    save("dgl_simple_var", dict(kind="dgl_simple", h=h, edge_index=ei, avg_d=avg_d, aggregators=aggr, scalers=scal,
                                ctor=dict(in_dim=f, out_dim=f, dropout=0.0, batch_norm=True, residual=True, posttrans_layers=1),
                                state_dict=lay.state_dict(), aggregate=agg, out=out))
    # dense layer, self_loop=True, aggregators incl. var, directed 0/1 adjacency without empty rows or columns
    torch.manual_seed(22)
    B, n, f = 2, 14, 8
    adj = (torch.rand(B, n, n) < 0.25).float()
    adj = adj * (1 - torch.eye(n))                       # the layer adds the loop itself
    for b in range(B):
        for i in range(n):
            if adj[b, i].sum() == 0:
                adj[b, i, (i + 1) % n] = 1
            if adj[b, :, i].sum() == 0:
                adj[b, (i + 2) % n, i] = 1
    table = torch.rand(3, f)
    hd = table[torch.randint(0, 3, (B, n))]
    hd[:, ::3] = torch.rand(B, (n + 2) // 3, f)         # a mix of identical and distinct rows
    avg_dd = dict(lin=adj.sum(-1).mean().item(), log=torch.log(adj.sum(-1) + 1).mean().item())
    aggrs = ["mean", "max", "min", "std", "var"]
    for name, loop in (("dense_self_loop", True), ("dense_directed", False)):
        layd = DensePNALayer(f, f, aggrs, S3, avg_dd, towers=2, self_loop=loop, pretrans_layers=1, posttrans_layers=1,
                             divide_input=True)
        layd.eval()
        with torch.no_grad():
            outd = layd(hd, adj)
        save(name, dict(kind="dense", adj=adj, h=hd, avg_d=avg_dd, aggregators=aggrs, scalers=S3,
                        ctor=dict(in_features=f, out_features=f, towers=2, self_loop=loop, pretrans_layers=1,
                                  posttrans_layers=1, divide_input=True), state_dict=layd.state_dict(), out=outd))


def propagate_case():
    """PNAConvSimple.propagate alone on a random multigraph, example.py's aggregator order: the aggregation the oracle
    restates, pinned bit for bit by tests/test_oracle.py."""
    torch.manual_seed(5)
    n, e, f = 300, 2000, 24
    x = torch.randn(n, f)
    ei = torch.randint(0, n, (2, e))
    deg = deg_hist(ei[1], n)
    conv = PNAConvSimple(f, f, A4_EX, S3, deg)
    with torch.no_grad():
        agg = conv.propagate(ei, x=x, size=None)
    save("pyg_propagate_f24", dict(kind="pyg_propagate", x=x, edge_index=ei, deg=deg, aggregators=A4_EX, scalers=S3,
                                   avg_deg=conv.avg_deg, aggregate=agg))


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    if "--round2" in sys.argv:
        round2_cases()
        sys.exit(0)
    if "--propagate" in sys.argv:
        propagate_case()
        sys.exit(0)
    simple_case("pyg_simple_f16", 200, 900, 16, seed=1)
    simple_case("pyg_simple_f64_hub", 100, 400, 64, seed=2, hub=700)
    simple_case("pyg_simple_f75_const", 90, 260, 75, seed=3, aggrs=A4_EX, constant_rows=True)
    simple_case("pyg_simple_allops", 80, 300, 12, seed=4, aggrs=["sum", "mean", "min", "max", "var", "std"],
                scalers=["identity", "amplification", "attenuation", "linear", "inverse_linear"], post_layers=2)
    conv_case("pyg_conv_t1", 100, 420, 32, 32, seed=5)
    conv_case("pyg_conv_t4_div", 100, 420, 32, 32, seed=6, towers=4, divide_input=True, post_layers=2)
    conv_case("pyg_conv_t5_rep", 80, 300, 15, 20, seed=7, towers=5, divide_input=False)
    conv_case("pyg_conv_edge", 80, 300, 16, 16, seed=8, towers=2, divide_input=True, edge_dim=5)
    conv_case("pyg_conv_pre2", 80, 300, 16, 16, seed=9, towers=2, divide_input=False, pre_layers=2)
    multitask_case()
    dgl_cases()
    dense_and_numpy_cases()
