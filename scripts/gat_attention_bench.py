"""GATConv with ``return_attention_weights`` on a C5-style graph: the cost of asking for alpha, timed with CUDA events.

    python scripts/gat_attention_bench.py --out RESULTS.jsonl [--iters 20] [--warmup 5]

Graph: 256 graphs x 2000 nodes, kNN-8 (E = 4.1M), F_in = 256, H*C = 256 with (H, C) = (1, 256) and (8, 32), concat.  Per
configuration, layer forward + backward:
  - ``plain``: ``layer(x, ei)``, loss on out (heads = 1 runs ``gat_conv``, heads = 8 ``gat_conv_heads``);
  - ``alpha_out_loss``: ``layer(x, ei, return_attention_weights=True)``, loss on out only;
  - ``alpha_both_loss``: the same with a loss on out and on alpha (the alpha gradient enters ``dc_gat_bwd_edge_heads_ext``);
and the by-receiver backward kernel alone: ``dc_gat_bwd_edge_heads`` against ``dc_gat_bwd_edge_heads_ext`` with both alpha
gradients given, on the same inputs.  The working sets (xs 537 MB, alpha up to 147 MB) exceed the 126 MB L2; no explicit flush
between iterations.  Writes one JSON line per configuration plus one line with the card, its power limit and SM clocks
(query-only nvidia-smi).
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

CONFIGS = [(1, 256, True), (8, 32, True)]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    name, power, max_clock, clock = [s.strip() for s in q.split(",")] if q.count(",") == 3 else (q, "", "", "")
    return {"gpu": name, "power_limit": power, "max_sm_clock": max_clock, "sm_clock": clock,
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSON-lines file to write")
    ap.add_argument("--graphs", type=int, default=256)
    ap.add_argument("--nodes", type=int, default=2000)
    ap.add_argument("--k", type=int, default=8)
    ap.add_argument("--fin", type=int, default=256)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("gat_attention_bench.py measures on a CUDA device; none found")
    import deformcontact_b200 as dc
    from deformcontact_b200 import _abi, ops

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    B, n, k, fin = args.graphs, args.nodes, args.k, args.fin
    N = B * n
    gen = torch.Generator(device=dev).manual_seed(0)
    pos = torch.rand(N, 3, generator=gen, device=dev) - 0.5
    ei = dc.knn_graph(pos, k, ptr=torch.arange(B + 1, device=dev) * n)
    E = int(ei.shape[1])
    x = torch.randn(N, fin, generator=gen, device=dev)
    g = ops.graph_csr(ei, N, "gat", None)
    _ = g.t
    keep, ei_sl = g.attention_edges()
    it, wu = args.iters, args.warmup
    E_nl = E if keep is None else int(keep.numel())
    lines = [dict(kind="setup", workload=f"{B} kNN-{k} graphs x {n} nodes, N={N}, E={E}, E_nl={E_nl}, F_in={fin}", iters=it,
                  warmup=wu, timing="CUDA events around `iters` back-to-back calls after `warmup` calls", **gpu_info())]
    st = torch.cuda.current_stream().cuda_stream
    p = lambda t: None if t is None else t.data_ptr()

    for H, C, concat in CONFIGS:
        torch.manual_seed(0)
        layer = dc.GATConv(fin, C, heads=H, concat=concat).to(dev)
        gout = torch.randn(N, H * C, generator=gen, device=dev)
        galpha = torch.randn(ei_sl.shape[1], H, generator=gen, device=dev)
        xg = x.clone().requires_grad_(True)

        def fb(mode):
            layer.zero_grad(set_to_none=True)
            xg.grad = None
            if mode == "plain":
                layer(xg, ei).backward(gout)
                return
            out, (_, alpha) = layer(xg, ei, return_attention_weights=True)
            if mode == "alpha_out_loss":
                out.backward(gout)
            else:
                torch.autograd.backward([out, alpha], [gout, galpha])

        rec = dict(kind="config", heads=H, C=C, concat=concat)
        for mode in ("plain", "alpha_out_loss", "alpha_both_loss"):
            rec[f"layer_fwd_bwd_ms_{mode}"] = ev_time(lambda: fb(mode), it, wu)
        rec["alpha_both_loss_overhead_ms"] = rec["layer_fwd_bwd_ms_alpha_both_loss"] - rec["layer_fwd_bwd_ms_plain"]

        with torch.no_grad():
            res = torch.ops.dcb200.gat_conv_heads(x, ei, layer.lin.weight, layer.att_src, layer.att_dst, layer.bias, 0.2, H, concat,
                                                  False, ops.GEMM_AUTO, None)
        _, xs, a_src, a_dst, alpha_e, alpha_s = res
        dalpha_e = torch.randn(alpha_e.shape, generator=gen, device=dev)
        dalpha_s = torch.randn(alpha_s.shape, generator=gen, device=dev)
        outs = (torch.zeros_like(alpha_e), torch.empty_like(alpha_s), torch.empty_like(alpha_s))
        hs, scale = ops._dout_heads(H, C, concat)
        common = (p(g.rowptr), p(g.nbr), p(g.eid), p(a_src), p(a_dst), 0.2, p(alpha_e), p(alpha_s), p(xs), xs.stride(0), p(gout),
                  gout.stride(0), hs, scale, H, C, N)
        base = lambda: _abi.call("dc_gat_bwd_edge_heads", *common, *[p(t) for t in outs], st)
        ext = lambda: _abi.call("dc_gat_bwd_edge_heads_ext", *common, p(dalpha_e), p(dalpha_s), *[p(t) for t in outs], st)
        rec["kernel_ms_dc_gat_bwd_edge_heads"] = ev_time(base, it, wu)
        rec["kernel_ms_dc_gat_bwd_edge_heads_ext"] = ev_time(ext, it, wu)
        rec["ext_kernel_extra_bytes"] = 4 * (E + N) * H      # the two alpha gradients, read once
        lines.append(rec)
        print(json.dumps(rec), flush=True)
        del layer, xg, res, xs, alpha_e, alpha_s, dalpha_e, dalpha_s, outs
        torch.cuda.empty_cache()

    info = gpu_info()
    lines.append(dict(kind="end", sm_clock_at_end=info["sm_clock"]))
    with open(args.out, "w") as f:
        for r in lines:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
