#!/usr/bin/env python
"""bench.py -- aggregated edges/s of the PNA layer forward on B200 (BASELINE.json metric), one JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over the whole graph: CSR (resident, built once) -> [N, 12*F] aggregation
(mean/max/min/std x identity/amplification/attenuation) -- the kernels of libpna_sm100.so and nothing else.
  value        edges/s of that step, inputs resident in HBM, CUDA events around each step, L2 flushed between steps
  e2e          edges/s of PNAConvSimple.forward(x, edge_index) called with pinned HOST tensors: H2D of x and
               edge_index, CSR build, aggregation, post-MLP, D2H of the layer output, all inside the timed region
  roofline     B_min (SURVEY.md 8d) / step time against MEASURED_PEAKS.json's HBM copy bandwidth
  parity       the step's output compared with the CPU oracle inside this run (every row at N = 1), asserted
  configs      (N = 1) the other BASELINE.json shapes that fit one GPU -- configs[0], [2], one GPU's share of [3] and [4] --
               each with its step time, B_min fraction and in-run parity; configs[0] also times the reference's CPU PNAConv
  cpu_baseline the reference's PyTorch CPU op sequence (oracle/pna_oracle.py, a port: torch_geometric/torch_scatter
               are not installable) timed on the host cores of this box on the same graph
N = 1: BASELINE.json configs[1] (ogbn-arxiv-shaped, 169 343 nodes / 1 166 243 edges, F = 128, fp32).
N > 1: bench_multi.py -- configs[3] at N = 4 (graph-batch shard), configs[4] at N = 8 (destination partition + halo exchange),
       configs[4] at N/8 scale otherwise.
--impl reference: the same workload's reference op sequence on the host cores (rank 0 only), same config / steps / warm-up.
--dump-outputs DIR (N = 1): DIR/aggregate.npy, float32 rows of the last timed step's [N, 12*F] output (dump_rows says which),
               so that two builds can be compared output for output on identical seeded inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench_common as bc                                   # noqa: E402
from bench_common import AGGRS, SCALERS, METRIC, UNIT        # noqa: E402


def config2_dict(n, e, f, max_deg):
    """Printed identically by both arms."""
    return {"workload": "ogbn-arxiv-shaped CSR (BASELINE.json configs[1])", "n_nodes": n, "n_edges": e, "n_feat": f,
            "aggregators": AGGRS, "scalers": SCALERS, "dst_skew": "perm[floor(N*u^3)]", "max_in_degree": max_deg,
            "l2": bc.L2_NOTE, "parallelism": "1 gpu"}


def best_thread_count(fn):
    """torch's CPU scatter/index kernels do not scale to 100+ threads (oversubscription makes them slower): a few thread
    counts are tried and the FASTEST is used -- the baseline gets every advantage the hardware offers."""
    ncpu = os.cpu_count() or 1
    candidates = sorted({ncpu, min(ncpu, 64), min(ncpu, 32), min(ncpu, 16), min(ncpu, 8)}, reverse=True)
    best_t, best_n = None, ncpu
    for n in candidates:
        torch.set_num_threads(n)
        fn()
        t0 = time.perf_counter()
        fn()
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best_t, best_n = dt, n
    torch.set_num_threads(best_n)
    return best_n, {"threads_tried": candidates, "host_cpus": ncpu}


def cpu_time(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return ts


# ---- --impl reference ----------------------------------------------------------------------------------------------------
def reference_workload(world: int):
    """(edge_index, x, config dict, sample note) of the reference arm: the workload of the repo arm at this N, bounded so
    that one CPU pass takes about a second (N = 1: the full config-2 graph)."""
    from pna_b200 import synth
    import bench_multi
    if world == 1:
        ei, x = synth.arxiv_like(n_feat=128, seed=0)
        md = int(torch.bincount(ei[1], minlength=x.size(0)).max())
        return ei, x, config2_dict(x.size(0), ei.size(1), 128, md), 1.0, "full config-2 graph"
    cfg = bench_multi.config_dict(world)
    if bench_multi.workload_for(world) == "config4":
        ei = synth.superpixel_shard(0, 2500, "cpu")
        x = synth.hash_features(torch.arange(2500 * 70), 64)
        return ei, x, cfg, 2500 * 70 * 8 / cfg["n_edges"], "2 500 of the 60 000 superpixel graphs (175 000 nodes / 1.4 M edges, F=64)"
    n, e, f = 156_250, 1_562_500, cfg["n_feat"]
    src, dst = next(iter(synth.powerlaw_stream(n, e, "cpu", seed=0, chunk=e)))
    x = synth.hash_features(torch.arange(n), f)
    return torch.stack([src, dst]), x, cfg, e / cfg["n_edges"], \
        f"a 1/{cfg['n_edges'] // e} scale instance of the power-law generator (156 250 nodes / 1 562 500 edges, F={f})"


def run_reference(args):
    """--impl reference: the reference arm (CPU).  Under torchrun only rank 0 works."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from pna_b200 import synth
    from oracle import pna_oracle as O
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    world = max(world, args.gpus)
    ei, x, cfg, frac, sample = reference_workload(world)
    n, e, f = x.size(0), ei.size(1), x.size(1)
    deg = synth.degree_histogram(ei[1], n)
    avg = O.avg_deg_from_histogram(deg)
    torch.manual_seed(0)
    lay = O.PNAConvSimpleOracle(f, f, AGGRS, SCALERS, deg)
    with torch.no_grad():
        threads, info = best_thread_count(lambda: O.simple_propagate(x, ei, AGGRS, SCALERS, avg))
        ts = cpu_time(lambda: O.simple_propagate(x, ei, AGGRS, SCALERS, avg), args.steps, args.warmup)
        tl = cpu_time(lambda: lay(x, ei), max(2, min(args.steps, 5)), 1)
    v = e * len(ts) / sum(ts)
    v_layer = e * len(tl) / sum(tl)
    what = ("the reference's aggregation op sequence (index_select, 6x scatter_add, amin, amax, degree, 3 scalers, cats: "
            "models/pytorch_geometric/pna.py:242-249, aggregators.py, scalers.py restated in oracle/pna_oracle.py) in torch CPU")
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": len(ts), "warmup": args.warmup,
        "ms_per_step": 1e3 * sum(ts) / len(ts), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port", **info,
                         "sample": f"{sample}: {len(ts)} passes of {what}", "sample_fraction_of_workload": frac},
        "e2e": {"value": v_layer, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "what": "PNAConvSimple.forward (aggregation + post-MLP Linear) on the same sample, torch CPU"},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---- the other single-GPU shapes (N = 1 `configs`) ------------------------------------------------------------------------
def side_configs(dev, flush, steps, peak):
    import pna_b200
    from pna_b200 import synth
    from oracle import pna_oracle as O
    res = {}

    def measure(name, src, dst, x, features_of, note, n_sample, extra=None):
        n, f = x.shape
        e = int(src.numel())
        deg_hist = torch.bincount(torch.bincount(dst, minlength=n)).cpu()
        avg = pna_b200.avg_deg_from_histogram(deg_hist)
        csr = pna_b200.build_csr(src.to(dev), dst.to(dev), n)
        xd = x.to(dev)
        out = torch.empty((n, 12 * f), dtype=x.dtype, device=dev)
        ts = bc.timed_steps(lambda: pna_b200.aggregate_forward(xd, csr, AGGRS, SCALERS, avg, out=out), steps, 3, flush)
        ms = sum(ts) / len(ts)
        par = bc.sampled_parity(out, csr.rowptr, csr.col, features_of, avg, csr.split_threshold, n_rows_sample=n_sample,
                                max_edges=4_000_000, rows=_rows_with_hubs(csr, n_sample))
        by = synth.algorithmic_bytes(n, e, f, x.element_size(), 12 * f)
        rec = {"workload": note, "n_nodes": n, "n_edges": e, "n_feat": f, "dtype": str(x.dtype).replace("torch.", ""), "ms_per_step": ms,
               "edges_per_s": e / (ms * 1e-3), "b_min_bytes": by["b_min"], "frac_of_measured_hbm_peak": by["b_min"] / (ms * 1e-3) / 1e9 / peak,
               "split_rows": csr.n_hubs, "max_in_degree": csr.max_degree, "parity_ok": par["ok"],
               "parity_max_err": max(par["max_err_light"], par["max_err_split_vs_f64"]), "parity_max_err_over_tolerance": par["max_err_over_tol"],
               "parity_rows": par["rows"] + par["big_rows"],
               "parity_rows_are_all_rows": par["rows"] + par["big_rows"] == n}
        if extra:
            rec.update(extra(csr, xd, avg, deg_hist))
        res[name] = rec
        assert par["ok"], f"parity failed on {name}: {par}"
        del out, xd, csr
        torch.cuda.empty_cache()

    # configs[0]: 64 x 1k-node graphs, F = 16; plus the reference's own CPU PNAConv(16,16,towers=4,divide_input=True) timing
    ei, x = synth.multitask_like()

    def config1_layer(csr, xd, avg, deg_hist):
        torch.manual_seed(0)
        ref = O.PNAConvOracle(16, 16, AGGRS, SCALERS, deg_hist, towers=4, divide_input=True)
        lay = pna_b200.PNAConv(16, 16, AGGRS, SCALERS, deg_hist, towers=4, divide_input=True)
        lay.load_state_dict(ref.state_dict())
        lay = lay.to(dev)
        eid = ei.to(dev)
        with torch.no_grad():
            threads, info = best_thread_count(lambda: ref(x, ei))
            tc = cpu_time(lambda: ref(x, ei), 3, 1)
            want = ref(x, ei)
            got = lay(xd, eid, csr=csr)
            for _ in range(3):
                lay(xd, eid, csr=csr)
            s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(20):
                lay(xd, eid, csr=csr)
            t.record(); torch.cuda.synchronize()
        err = float((got.cpu() - want).abs().max())
        cpu_ms = 1e3 * sum(tc) / len(tc)
        gpu_ms = s.elapsed_time(t) / 20
        return {"layer": "PNAConv(16, 16, towers=4, divide_input=True) forward (multitask_benchmark/README.md:36)",
                "cpu_reference": {"ms": cpu_ms, "edges_per_s": ei.size(1) / (cpu_ms * 1e-3), "cores": threads, "kind": "port", **info,
                                  "what": "the reference's PNAConv op sequence (oracle/pna_oracle.py PNAConvOracle) in torch CPU, 3 passes"},
                "gpu_layer": {"ms": gpu_ms, "edges_per_s": ei.size(1) / (gpu_ms * 1e-3), "max_abs_err_vs_cpu_reference": err}}
    measure("configs[0]", ei[0], ei[1], x, lambda idx: x[idx], "multitask-shaped batch: 64 x 1 000-node random graphs, F=16 fp32",
            64_000, config1_layer)

    # configs[2]: ZINC-shaped batch, F = 75 bf16 (unpadded 150-byte rows)
    ei, x, _ = synth.zinc_like(dtype=torch.bfloat16)
    def config3_as_the_layers_run_it(csr, xd, avg, deg_hist):
        """The layers never call the kernel on 150-byte rows: they run F=75 at feature pitch 80 (zero pad columns, absorbed by
        zero columns of the first post Linear; pna_b200/padding.py).  Same graph, same step, B_min still counted for F=75;
        the valid columns must equal the unpadded call's bit for bit."""
        n = xd.size(0)
        x80 = torch.nn.functional.pad(xd, (0, 5))
        out80 = torch.empty((n, 12 * 80), dtype=xd.dtype, device=dev)
        ts = bc.timed_steps(lambda: pna_b200.aggregate_forward(x80, csr, AGGRS, SCALERS, avg, out=out80), steps, 3, flush)
        ms = sum(ts) / len(ts)
        out75 = pna_b200.aggregate_forward(xd, csr, AGGRS, SCALERS, avg)
        same = bool(torch.equal(out80.view(n, 12, 80)[:, :, :75].reshape(n, 900), out75))
        by = synth.algorithmic_bytes(n, csr.n_edges, 75, 2, 12 * 75)
        return {"at_feature_pitch_80": {"ms_per_step": ms, "edges_per_s": csr.n_edges / (ms * 1e-3),
                                        "frac_of_measured_hbm_peak": by["b_min"] / (ms * 1e-3) / 1e9 / peak,
                                        "valid_columns_equal_unpadded_call": same,
                                        "what": "x and out at pitch 80 (how PNAConvSimple / PNASimpleLayer run odd widths); "
                                                "B_min counted for F=75"}}
    measure("configs[2]", ei[0], ei[1], x, lambda idx: x[idx], "ZINC-shaped batch: 12 000 molecule-like graphs, F=75 bf16 (150-byte rows)",
            x.size(0), config3_as_the_layers_run_it)

    # the ZINC-shaped full layer (realworld_benchmark/configs: towers=5, 75 -> 75): PNAConv forward, fp32, CSR cached
    ei32, x32, _ = synth.zinc_like(dtype=torch.float32)
    degh = synth.degree_histogram(ei32[1], x32.size(0))
    torch.manual_seed(0)
    refl = O.PNAConvOracle(75, 75, AGGRS, SCALERS, degh, towers=5, divide_input=True)
    layl = pna_b200.PNAConv(75, 75, AGGRS, SCALERS, degh, towers=5, divide_input=True)
    layl.load_state_dict(refl.state_dict())
    layl = layl.to(dev)
    xl, eil = x32.to(dev), ei32.to(dev)
    csrl = pna_b200.build_csr(eil[0], eil[1], x32.size(0))
    with torch.no_grad():
        wantl = refl(x32, ei32)
        gotl = layl(xl, eil, csr=csrl)
        for _ in range(3):
            layl(xl, eil, csr=csrl)
        s_, t_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s_.record()
        for _ in range(20):
            layl(xl, eil, csr=csrl)
        t_.record(); torch.cuda.synchronize()
    res["configs[2] layer"] = {"workload": "ZINC-shaped batch, PNAConv(75, 75, towers=5, divide_input=True) forward, fp32, CSR cached",
                               "n_nodes": x32.size(0), "n_edges": ei32.size(1), "ms": s_.elapsed_time(t_) / 20,
                               "edges_per_s": ei32.size(1) / (s_.elapsed_time(t_) / 20 * 1e-3),
                               "max_abs_err_vs_cpu_reference": float((gotl.cpu() - wantl).abs().max())}
    del xl, eil, csrl, layl, gotl
    torch.cuda.empty_cache()

    # configs[3], one GPU's share: 15 000 superpixel graphs, F = 64
    ei = synth.superpixel_shard(0, 15_000, dev)
    n4 = 15_000 * 70
    x4 = synth.hash_features(torch.arange(n4, device=dev), 64)
    measure("configs[3] (one GPU's share)", ei[0], ei[1], x4, lambda idx: synth.hash_features(idx, 64),
            "15 000 of the 60 000 superpixel kNN graphs (70 nodes, k=8), F=64 fp32", 120_000)
    del x4

    # configs[4], one GPU's share: power-law 1.25 M / 12.5 M, F = 256
    src, dst = next(iter(synth.powerlaw_stream(1_250_000, 12_500_000, dev, seed=0)))
    x5 = synth.hash_features(torch.arange(1_250_000, device=dev), 256)
    measure("configs[4] (one GPU's share)", src, dst, x5, lambda idx: synth.hash_features(idx, 256),
            "power-law 1.25 M nodes / 12.5 M edges (Zipf 1.5 sources and destinations), F=256 fp32", 100_000)
    return res


DUMP_LIMIT_BYTES = 64_000_000          # everything --dump-outputs writes, .npy header included


def dump_rows(rowptr, row_bytes):
    """Rows of the step's output that --dump-outputs writes: the whole output when it fits DUMP_LIMIT_BYTES, otherwise the
    64 rows of largest in-degree (split across warps) plus a seeded random sample of the others, sorted.  A function of
    the graph only, so every build writes the same rows."""
    n = rowptr.numel() - 1
    k = min(n, (DUMP_LIMIT_BYTES - 128) // row_bytes)
    deg = (rowptr[1:] - rowptr[:-1]).cpu()
    heavy = torch.sort(deg, descending=True, stable=True).indices[:min(64, k)]
    rest = torch.randperm(n, generator=torch.Generator().manual_seed(0))
    rest = rest[~torch.isin(rest, heavy)][:k - heavy.numel()]
    return torch.sort(torch.cat([heavy, rest])).values


def _rows_with_hubs(csr, n_sample):
    g = torch.Generator().manual_seed(11)
    rows = torch.randperm(csr.n_nodes, generator=g)[: min(n_sample, csr.n_nodes)]
    if csr.n_hubs and n_sample < csr.n_nodes:
        info = csr.hub_info.cpu().long()
        rows = torch.unique(torch.cat([rows, info[torch.argsort(info[:, 3], descending=True)[:16], 0]]))
    return rows


# ---- the repo arm at N = 1 ----------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist
    import pna_b200
    from pna_b200 import synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch N > 1 with torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1 or os.environ.get("PNA_BENCH_FORCE_MULTI") == "1":     # (the latter: exercise bench_multi.py on one GPU)
        if world == 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1"); os.environ.setdefault("MASTER_PORT", "29599")
            os.environ.setdefault("RANK", "0"); os.environ.setdefault("WORLD_SIZE", "1")
        dist.init_process_group("nccl", device_id=dev)
        import bench_multi
        return bench_multi.run(args)

    ei, x = synth.arxiv_like(n_feat=128, seed=0)
    n, e, f = x.size(0), ei.size(1), x.size(1)
    deg_hist = synth.degree_histogram(ei[1], n)
    avg_deg = pna_b200.avg_deg_from_histogram(deg_hist)
    xd, eid = x.to(dev), ei.to(dev)

    # CSR: once per graph (cached by the layers); timed separately
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    csr = pna_b200.build_csr(eid[0], eid[1], n)
    torch.cuda.synchronize()
    csr_ms_first = 1e3 * (time.perf_counter() - t0)
    for _ in range(3):
        pna_b200.build_csr(eid[0], eid[1], n)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ev[0].record()
    for _ in range(5):
        pna_b200.build_csr(eid[0], eid[1], n)
    ev[1].record()
    torch.cuda.synchronize()
    csr_ms = ev[0].elapsed_time(ev[1]) / 5
    csr_wall_ms = 1e3 * (time.perf_counter() - t0) / 5

    out = torch.empty((n, 12 * f), dtype=torch.float32, device=dev)
    flush = bc.L2Flush(dev)

    def step(**kw):
        pna_b200.aggregate_forward(xd, csr, AGGRS, SCALERS, avg_deg, out=out, **kw)

    # clocks / throttle reasons are sampled (20 Hz) while the GPU runs this workload: the timed steps themselves last
    # only ~15 ms, so the sampler brackets them with extra untimed passes of the same kernels to collect enough samples
    with bc.ClockSampler(local) as clk:
        time.sleep(0.06)
        t_end = time.perf_counter() + 0.5
        while time.perf_counter() < t_end:
            step()
        torch.cuda.synchronize()
        per_step = bc.timed_steps(step, args.steps, args.warmup, flush)
        if args.dump_outputs:                       # before the untimed passes below overwrite `out`
            dumped = out[dump_rows(csr.rowptr, out.size(1) * out.element_size()).to(dev)].cpu()
        t_end = time.perf_counter() + 0.5
        while time.perf_counter() < t_end:
            step()
        torch.cuda.synchronize()
    clocks = clk.summary()
    t_ms = sum(per_step) / len(per_step)
    value = e / (t_ms * 1e-3)
    from pna_b200.aggregate import fold_finalize_enabled
    launches_per_step = 1 + (1 if (csr.n_hubs and not fold_finalize_enabled()) else 0)

    # in-run parity: EVERY row of the step's output against the CPU oracle
    par = bc.sampled_parity(out, csr.rowptr, csr.col, lambda idx: x[idx], avg_deg, csr.split_threshold, n_rows_sample=n,
                            max_edges=1 << 40, rows=torch.arange(n))
    assert par["ok"], f"parity failed: {par}"

    bytes_ = synth.algorithmic_bytes(n, e, f, 4, 12 * f)
    peak, peak_src = bc.measured_peaks()
    achieved = bytes_["b_min"] / (t_ms * 1e-3) / 1e9
    traffic = None
    prof = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(prof):
        try:
            traffic = json.load(open(prof)).get("dram_bytes_per_step")
        except Exception:
            traffic = None

    # e2e: the public layer call with HOST buffers (pinned), copies inside the timed region
    torch.manual_seed(0)
    lay = pna_b200.PNAConvSimple(f, f, AGGRS, SCALERS, deg_hist).to(dev)
    xh = x.pin_memory()
    outh = torch.empty((n, f), dtype=torch.float32).pin_memory()
    eih_steps = [ei.clone().pin_memory() for _ in range(4)]    # distinct host tensors: the device copy is always fresh

    def e2e_step():
        # the public host-buffer call: pinned x / edge_index in, pinned result out; a new edge_index object every step,
        # so the CSR is rebuilt inside the call (nothing is cached across steps)
        lay.forward_host(xh, eih_steps[e2e_step.i % len(eih_steps)], out=outh)
        e2e_step.i += 1
    e2e_step.i = 0

    # PCIe health of this box (context for e2e: the layer call moves 192 MB per step over PCIe)
    def copy_rate(fn, nbytes):
        fn(); torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize()
        return nbytes / (a.elapsed_time(b) * 1e-3) / 1e9
    xdev_tmp = torch.empty_like(xd)
    h2d_gbs = copy_rate(lambda: xdev_tmp.copy_(xh, non_blocking=True), xh.numel() * 4)
    ydev_tmp = torch.empty((n, f), dtype=torch.float32, device=dev)
    d2h_gbs = copy_rate(lambda: outh.copy_(ydev_tmp, non_blocking=True), n * f * 4)
    del xdev_tmp, ydev_tmp

    k2 = max(3, min(args.steps, 20))
    for _ in range(3):
        e2e_step()
    torch.cuda.synchronize()
    s2, e2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    s2.record()
    for _ in range(k2):
        e2e_step()
    e2.record()
    torch.cuda.synchronize()
    e2e_wall_ms = 1e3 * (time.perf_counter() - t0) / k2
    e2e_ms = max(s2.elapsed_time(e2) / k2, e2e_wall_ms)      # host-side launch/sync time counts too

    def layer_ms():
        with torch.no_grad():
            s3, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            for _ in range(3):
                lay(xd, eid, csr=csr)
            s3.record()
            for _ in range(20):
                lay(xd, eid, csr=csr)
            e3.record()
            torch.cuda.synchronize()
            return s3.elapsed_time(e3) / 20
    full_ms = layer_ms()                        # compact post path: [N, 4F] aggregate + pna_linear_scaled_fwd
    os.environ["PNA_B200_COMPACT_POST"] = "0"
    full_ms_12f = layer_ms()                    # the same layer through the materialised [N, 12F] tensor
    del os.environ["PNA_B200_COMPACT_POST"]

    cpu = None
    if not args.no_cpu_baseline:
        from oracle import pna_oracle as O
        with torch.no_grad():
            threads, info = best_thread_count(lambda: O.simple_propagate(x, ei, AGGRS, SCALERS, avg_deg))
            tc = cpu_time(lambda: O.simple_propagate(x, ei, AGGRS, SCALERS, avg_deg), 3, 1)
        cpu = {"value": e * len(tc) / sum(tc), "unit": UNIT, "cores": threads, "kind": "port", **info,
               "sample": "full config-2 graph, 3 passes of the reference's aggregation op sequence (models/pytorch_geometric/pna.py:"
                         "242-249 restated in oracle/pna_oracle.py; torch_geometric/torch_scatter not installable) in torch CPU"}

    sides = None
    if not args.no_side_configs:
        del out
        torch.cuda.empty_cache()
        sides = side_configs(dev, flush, max(5, min(args.steps, 20)), peak)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": t_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": config2_dict(n, e, f, csr.max_degree),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "peak_source": peak_src, "bytes_model": "B_min = N*F*s + 4E + 4(N+1) + 12*N*F*s",
                     "b_min_bytes": bytes_["b_min"], "b_gather_bytes": bytes_["b_gather"],
                     "effective_gbs_b_gather": bytes_["b_gather"] / (t_ms * 1e-3) / 1e9},
        "parity": {"ok": par["ok"], "parity_max_err": max(par["max_err_light"], par["max_err_split_vs_f64"]),
                   "max_err_over_tolerance": par["max_err_over_tol"], "tolerance": "|d| <= 1e-5 + 1e-5 |want| (north star: 1e-5 fp32)",
                   "max_err_light_rows": par["max_err_light"], "max_err_split_rows_vs_f64": par["max_err_split_vs_f64"],
                   "rows_checked": par["rows"] + par["big_rows"], "split_rows_checked": par["split_rows"] + par["big_rows"],
                   "what": "every row of the timed step's output vs the CPU oracle (fp32 op sequence; rows split across warps vs float64)"},
        "kernels_ms": {"step_min": min(per_step), "step_median": statistics.median(per_step), "split_rows": csr.n_hubs,
                       "kernels": ("k_rows_stream (rows + chunks of split rows, split rows finalized by the last-arriving warp)"
                                   if fold_finalize_enabled() else "k_rows_stream (rows + chunks of split rows) + k_hub_finalize")
                                  + "; per-kernel times: profiles/"},
        "layer_fwd": {"ms": full_ms, "edges_per_s": e / (full_ms * 1e-3), "ms_via_12f_tensor": full_ms_12f,
                      "what": "PNAConvSimple.forward, CSR cached: aggregation with the identity scaler ([N,4F]) + post-MLP linear on "
                              "the tensor cores regenerating the scaled copies in registers (pna_linear_scaled_fwd, 3xTF32 "
                              "tcgen05); ms_via_12f_tensor = same layer through the materialised [N,12F] tensor"},
        "csr_build_ms": {"first_call": csr_ms_first, "steady": csr_ms, "steady_wall": csr_wall_ms},
        "e2e": {"value": e / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": x.numel() * 4 + ei.numel() * 8, "d2h_bytes_per_step": n * f * 4,
                "device_ms_per_step": s2.elapsed_time(e2) / k2, "wall_ms_per_step": e2e_wall_ms,
                "pcie_h2d_gbs": h2d_gbs, "pcie_d2h_gbs": d2h_gbs, "pinned": bool(xh.is_pinned() and outh.is_pinned()),
                "what": "PNAConvSimple.forward_host(x, edge_index) with pinned host tensors: H2D (x overlapped with the CSR build) + "
                        "aggregate + post-MLP in row blocks overlapped with the D2H of the result; CSR rebuilt every step"},
        "gpu_launches": launches_per_step * args.steps,
        "clocks": clocks,
        "cpu_baseline": cpu,
        "configs": sides,
    }
    if args.dump_outputs:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "aggregate.npy"), dumped.numpy())
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU leg (profiling runs)")
    ap.add_argument("--no-side-configs", action="store_true", help="skip the `configs` sub-object (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write rows of the last timed step's output to DIR/aggregate.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.gpus != 1):
        ap.error("--dump-outputs: --impl ours on one GPU only")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    main()
