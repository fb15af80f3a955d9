"""CPU checks of the host logic the multi-GPU bench relies on: the pull plan (no id exchange), the node-id hash features,
the device generators' shard independence, and the in-run parity checker itself (it must accept the oracle's own output and
reject a corrupted one)."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

A4 = ["mean", "max", "min", "std"]
S3 = ["identity", "amplification", "attenuation"]


def _graph(n=300, e=4000, seed=3):
    g = torch.Generator().manual_seed(seed)
    src = torch.randint(0, n, (e,), generator=g)
    dst = torch.randint(0, int(n * 0.9), (e,), generator=g)
    dst[: e // 4] = 11
    return src, dst


def test_pull_plan_reproduces_the_whole_graph_result():
    """Every rank's [local ; halo] graph, fed with the TRUE rows of its halo ids, gives the oracle's rows of that range."""
    from oracle import pna_oracle as O
    from pna_b200 import dist as pd, synth
    src, dst = _graph()
    n, f, world = 300, 5, 3
    x = synth.hash_features(torch.arange(n), f)
    deg = torch.bincount(dst, minlength=n)
    bounds = pd.partition_bounds(deg, world)
    avg = O.avg_deg_from_histogram(torch.bincount(deg))
    want = O.simple_propagate(x, torch.stack([src, dst]), A4, S3, avg)
    remote_total = 0
    for r in range(world):
        lo, hi = int(bounds[r]), int(bounds[r + 1])
        mine = (dst >= lo) & (dst < hi)
        plan = pd.build_pull_plan(src[mine], dst[mine], bounds, r, world)
        assert plan.n_local == hi - lo and plan.halo_ids.numel() == plan.n_halo == plan.enc.numel()
        # enc names (owner, row-on-owner) of every halo row
        own = plan.enc.long() >> plan.shift
        row = plan.enc.long() & ((1 << plan.shift) - 1)
        assert torch.equal(bounds[own] + row, plan.halo_ids)
        assert bool(((plan.halo_ids < lo) | (plan.halo_ids >= hi)).all())
        x_ext = torch.cat([x[lo:hi], x[plan.halo_ids]])
        got = O.simple_propagate(x_ext, torch.stack([plan.src_ext, plan.dst_local]), A4, S3, avg)[: plan.n_local]
        assert torch.equal(got, want[lo:hi])
        remote_total += plan.n_remote_edges
    assert remote_total == int(((pd.owner_of(src, bounds) != pd.owner_of(dst, bounds))).sum())


def test_hash_features_are_a_function_of_the_node_id_only():
    from pna_b200 import synth
    a = synth.hash_features(torch.arange(1000), 24)
    idx = torch.tensor([5, 999, 0, 5])
    assert torch.equal(synth.hash_features(idx, 24), a[idx])
    assert torch.equal(synth.hash_features(torch.arange(1000), 24, chunk=7), a)
    assert a.abs().max() < 1 and abs(float(a.mean())) < 0.02 and 0.5 < float(a.std()) < 0.65
    assert torch.equal(synth.hash_features(idx, 24, dtype=torch.bfloat16), a[idx].to(torch.bfloat16))


def test_superpixel_shards_do_not_depend_on_the_number_of_ranks():
    from pna_b200 import synth
    whole = synth.superpixel_shard(0, 40, "cpu", chunk=10)
    a = synth.superpixel_shard(0, 20, "cpu", chunk=10)
    b = synth.superpixel_shard(20, 20, "cpu", chunk=10)
    assert torch.equal(torch.cat([a, b + 20 * 70], 1), whole)
    assert whole.size(1) == 40 * 70 * 8 and int(whole.max()) == 40 * 70 - 1


def test_parity_checker_accepts_the_oracle_and_rejects_a_corrupted_row():
    """bench_common.sampled_parity against rows produced by the oracle itself (CPU tensors stand in for the device)."""
    import bench_common as bc
    from oracle import pna_oracle as O
    from pna_b200 import synth
    src, dst = _graph(n=400, e=9000, seed=9)
    n, f = 400, 6
    x = synth.hash_features(torch.arange(n), f)
    order = torch.sort(dst, stable=True).indices
    deg = torch.bincount(dst, minlength=n)
    rowptr = torch.cat([torch.zeros(1, dtype=torch.long), torch.cumsum(deg, 0)]).to(torch.int32)
    col = src[order].to(torch.int32)
    avg = O.avg_deg_from_histogram(torch.bincount(deg))
    out = O.simple_propagate(x, torch.stack([src, dst]), A4, S3, avg)
    kw = dict(avg_deg=avg, split_threshold=256, n_rows_sample=n, max_edges=1 << 30, rows=torch.arange(n))
    # the hub (row 11, 2 250+ in-edges) goes through the float64 branch, the rest through the fp32 branch
    res = bc.sampled_parity(out, rowptr, col, lambda idx: x[idx], **kw)
    assert res["ok"] and res["rows"] == n and res["split_rows"] >= 1 and res["max_err_light"] == 0.0
    # streamed float64 branch for very large rows
    res = bc.sampled_parity(out, rowptr, col, lambda idx: x[idx], big_row_edges=1000, big_row_cols=4, **kw)
    assert res["ok"] and res["big_rows"] == 1
    bad = out.clone()
    bad[37, 3] += 1e-3
    assert not bc.sampled_parity(bad, rowptr, col, lambda idx: x[idx], **kw)["ok"]
    bad = out.clone()
    bad[11, 2] += 1e-2
    assert not bc.sampled_parity(bad, rowptr, col, lambda idx: x[idx], big_row_edges=1000, big_row_cols=4, **kw)["ok"]
    # wrong source features (what a broken halo exchange would look like) are caught too
    assert not bc.sampled_parity(out, rowptr, col, lambda idx: x[(idx + 1) % n], **kw)["ok"]


def test_dump_rows_are_fixed_include_the_heaviest_and_fit_the_limit():
    """bench.py --dump-outputs: every row when the output fits, else a fixed sample holding the 64 largest in-degrees."""
    import bench
    src, dst = _graph()
    n = 300
    deg = torch.bincount(dst, minlength=n)
    rowptr = torch.cat([torch.zeros(1, dtype=torch.long), torch.cumsum(deg, 0)])
    assert torch.equal(bench.dump_rows(rowptr, 4 * 1536), torch.arange(n))
    row_bytes = bench.DUMP_LIMIT_BYTES // 100
    rows = bench.dump_rows(rowptr, row_bytes)
    assert rows.numel() == 99 and rows.numel() * row_bytes + 128 <= bench.DUMP_LIMIT_BYTES
    assert torch.equal(rows, torch.unique(rows)) and torch.equal(rows, bench.dump_rows(rowptr, row_bytes))
    heavy = torch.sort(deg, descending=True, stable=True).indices[:64]
    assert bool(torch.isin(heavy, rows).all()) and 11 in rows.tolist()
