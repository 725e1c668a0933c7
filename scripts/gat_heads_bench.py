"""Multi-head GATConv on a C5-style graph: the layer, each new K6 kernel and two baselines, timed with CUDA events.

    python scripts/gat_heads_bench.py --out RESULTS.jsonl [--iters 20] [--warmup 5]

Graph: 256 graphs x 2000 nodes, kNN-8 (E = 4.1M), F_in = 256.  Configurations (H, C): (1, 256), (2, 128), (4, 64), (8, 32) with
concat and (4, 64) with mean; H*C = 256 throughout, so every configuration moves the same feature bytes.  (1, 256) is timed twice:
through the layer (heads = 1: scores, dc_gat_softmax, dc_spmm) and through the multi-head op (``gat_conv_heads``).
Baselines, same process and inputs:
  (a) the oracle GATConv (stock PyTorch CUDA kernels, TF32 off); for the mean, its bias-free concat output averaged over the
      heads, + bias (PyG's concat=False);
  (b) the aggregation composed from existing kernels: H launches of dc_spmm, one per head's column slice, with that head's alpha
      column made contiguous outside the timed region.  It does not include the softmax, nor, for the mean, the average over
      heads, both of which dc_gat_aggregate does in the same launch.
The working sets (xs 537 MB, alpha up to 131 MB) exceed the 126 MB L2; no explicit flush between iterations.
Writes one JSON line per configuration plus one line with the card, its power limit and max SM clock (query-only nvidia-smi).
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

CONFIGS = [(1, 256, True), (2, 128, True), (4, 64, True), (8, 32, True), (4, 64, False)]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    name, power, max_clock, clock = [s.strip() for s in q.split(",")] if q.count(",") == 3 else (q, "", "", "")
    return {"gpu": name, "power_limit": power, "max_sm_clock": max_clock, "sm_clock_at_start": clock,
            "torch_device": torch.cuda.get_device_name(0)}


def ev_time(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def agg_bytes(N, E, H, C, concat):
    """Algorithmic HBM bytes of dc_gat_aggregate: xs read once (4NHC) and out written once (4N * width), per edge the neighbour
    and edge id (8) and the alpha row written (4H), per node rowptr (4), a_src / a_dst read and alpha_self written (12H).
    a_src gathers and alpha re-reads are assumed served from cache."""
    width = H * C if concat else C
    return 4 * N * H * C + 4 * N * width + E * (8 + 4 * H) + N * (4 + 12 * H)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSON-lines file to write")
    ap.add_argument("--graphs", type=int, default=256)
    ap.add_argument("--nodes", type=int, default=2000)
    ap.add_argument("--k", type=int, default=8)
    ap.add_argument("--fin", type=int, default=256)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--no-baseline-a", action="store_true", help="skip the oracle baseline (fast rehearsal)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("gat_heads_bench.py measures on a CUDA device; none found")
    import deformcontact_b200 as dc
    from deformcontact_b200 import ops
    import oracle

    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    info = gpu_info()
    B, n, k, fin = args.graphs, args.nodes, args.k, args.fin
    N = B * n
    gen = torch.Generator(device=dev).manual_seed(0)
    pos = torch.rand(N, 3, generator=gen, device=dev) - 0.5
    ei = dc.knn_graph(pos, k, ptr=torch.arange(B + 1, device=dev) * n)
    E = int(ei.shape[1])
    x = torch.randn(N, fin, generator=gen, device=dev)
    g = ops.graph_csr(ei, N, "gat", None)
    _ = g.t
    it, wu = args.iters, args.warmup
    lines = [dict(kind="setup", workload=f"{B} kNN-{k} graphs x {n} nodes, N={N}, E={E}, F_in={fin}", iters=it, warmup=wu,
                  timing="CUDA events around `iters` back-to-back calls after `warmup` calls", **info)]

    for H, C, concat in CONFIGS:
        HC, W = H * C, (H * C if concat else C)
        torch.manual_seed(0)
        layer = dc.GATConv(fin, C, heads=H, concat=concat).to(dev)
        gout = torch.randn(N, W, generator=gen, device=dev)
        xg = x.clone().requires_grad_(True)

        def fb(fwd):
            layer.zero_grad(set_to_none=True)
            xg.grad = None
            fwd(xg).backward(gout)

        rec = dict(kind="config", heads=H, C=C, concat=concat, out_width=W, alpha_saved_bytes=4 * E * H)
        via_layer = lambda inp: layer(inp, ei)
        rec["layer_fwd_ms"] = ev_time(lambda: via_layer(x), it, wu)
        rec["layer_fwd_bwd_ms"] = ev_time(lambda: fb(via_layer), it, wu)
        rec["layer_path"] = "gat_conv (heads=1)" if H == 1 else "gat_conv_heads"
        if H == 1:     # the same layer through the multi-head kernels
            via_heads = lambda inp: torch.ops.dcb200.gat_conv_heads(inp, ei, layer.lin.weight, layer.att_src, layer.att_dst, layer.bias,
                                                                    0.2, 1, True, False, ops.GEMM_AUTO, None)[0]
            rec["heads_op_fwd_ms"] = ev_time(lambda: via_heads(x), it, wu)
            rec["heads_op_fwd_bwd_ms"] = ev_time(lambda: fb(via_heads), it, wu)
            with torch.no_grad():
                rec["heads_op_out_bit_identical_to_layer"] = bool(torch.equal(via_heads(x), via_layer(x)))

        # the new kernels one by one, on the layer's own intermediates
        with torch.no_grad():
            out, xs, a_s, a_d, al_e, al_s = torch.ops.dcb200.gat_conv_heads(x, ei, layer.lin.weight, layer.att_src, layer.att_dst,
                                                                            layer.bias, 0.2, H, concat, False, ops.GEMM_AUTO, None)
        kern = {}
        kern["dc_gat_aggregate"] = ev_time(lambda: ops.gat_aggregate(g, xs, a_s, a_d, 0.2, H, C, concat, bias=layer.bias), it, wu)
        dz_e, dz_s, da_d = ops.gat_bwd_edge_heads(g, a_s, a_d, 0.2, al_e, al_s, xs, gout, H, C, concat)
        kern["dc_gat_bwd_edge_heads"] = ev_time(lambda: ops.gat_bwd_edge_heads(g, a_s, a_d, 0.2, al_e, al_s, xs, gout, H, C, concat),
                                                it, wu)
        att_s, att_d = layer.att_src.detach(), layer.att_dst.detach()
        _, da_s = ops.gat_scatter_heads(g, al_e, al_s, dz_e, dz_s, da_d, att_s, att_d, gout, H, C, concat)
        kern["dc_gat_scatter_heads"] = ev_time(lambda: ops.gat_scatter_heads(g, al_e, al_s, dz_e, dz_s, da_d, att_s, att_d, gout, H, C,
                                                                             concat), it, wu)
        kern["dc_gat_att_grad"] = ev_time(lambda: ops.gat_att_grad(xs, da_s, da_d, H, C), it, wu)
        rec["kernel_ms"] = kern
        nbytes = agg_bytes(N, E, H, C, concat)
        rec["aggregate_bytes"] = nbytes
        rec["aggregate_gbs"] = nbytes / (kern["dc_gat_aggregate"] * 1e-3) / 1e9

        # baseline (b): H dc_spmm launches over the heads' column slices (alpha columns made contiguous outside the timing)
        al_cols = [al_e[:, h].contiguous() for h in range(H)]
        as_cols = [al_s[:, h].contiguous() for h in range(H)]
        outb = torch.empty((N, HC), device=dev)

        def per_head_spmm():
            for h in range(H):
                ops.spmm(g.rowptr, g.nbr, xs[:, h * C:(h + 1) * C], edge_w=al_cols[h], edge_w_index=g.eid, self_w=as_cols[h],
                         self_loop=True, out=outb[:, h * C:(h + 1) * C])
        rec["baseline_b_per_head_spmm_ms"] = ev_time(per_head_spmm, it, wu)
        rec["aggregate_vs_b_speedup"] = rec["baseline_b_per_head_spmm_ms"] / kern["dc_gat_aggregate"]
        if concat:
            per_head_spmm()
            agg_nobias = ops.gat_aggregate(g, xs, a_s, a_d, 0.2, H, C, concat)[0]
            rec["baseline_b_bit_identical_to_aggregate"] = bool(torch.equal(outb, agg_nobias))
        del al_cols, as_cols, outb

        # baseline (a): the oracle layer on the same GPU, stock PyTorch kernels, fp32 (TF32 off)
        if not args.no_baseline_a:
            ref = oracle.GATConv(fin, C, heads=H, bias=concat).to(dev)
            ref.load_state_dict({k: v for k, v in layer.state_dict().items() if concat or k != "bias"})
            bias = layer.bias.detach().clone().requires_grad_(True)
            fwd_ref = (lambda inp: ref(inp, ei)) if concat else (lambda inp: ref(inp, ei).view(N, H, C).mean(dim=1) + bias)
            xr = x.clone().requires_grad_(True)

            def fb_ref():
                ref.zero_grad(set_to_none=True)
                xr.grad = bias.grad = None
                fwd_ref(xr).backward(gout)
            with torch.no_grad():
                rec["baseline_a_oracle_fwd_ms"] = ev_time(lambda: fwd_ref(x), it, wu)
            rec["baseline_a_oracle_fwd_bwd_ms"] = ev_time(fb_ref, it, wu)
            rec["layer_fwd_bwd_vs_a_speedup"] = rec["baseline_a_oracle_fwd_bwd_ms"] / rec["layer_fwd_bwd_ms"]
            with torch.no_grad():
                o_ref = fwd_ref(x)
                rec["layer_vs_oracle_rel_err"] = ((layer(x, ei) - o_ref).abs().max() / o_ref.abs().max()).item()
            del ref, xr, o_ref, bias
        del out, xs, a_s, a_d, al_e, al_s, dz_e, dz_s, da_d, da_s, layer, xg, gout
        torch.cuda.empty_cache()
        lines.append(rec)
        print(json.dumps(rec), flush=True)

    lines.append(dict(kind="clocks_at_end", **gpu_info()))
    with open(args.out, "w") as f:
        for r in lines:
            f.write(json.dumps(r) + "\n")
    print(json.dumps(lines[0]))


if __name__ == "__main__":
    main()
