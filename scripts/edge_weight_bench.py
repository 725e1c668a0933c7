"""TAGConv / GCNConv with PyG's edge_weight on the C5 graph: the layers, the two new kernels and a baseline, timed with CUDA events.

    python scripts/edge_weight_bench.py --out RESULTS.jsonl [--iters 20] [--warmup 5]

Graph: 256 graphs x 2000 nodes, kNN-8 (N = 512000, E = 4.1M), TAGConv(256, 256) and GCNConv(256, 256).  Per layer, fwd+bwd
(x requires grad) for three cases: edge_weight=None, weights U(0.1, 2) without grad, and the same weights with grad.
Kernels, on the layer's own intermediates: the weighted normalisation (dc_gcn_norm_weighted, both CSR orders, as the backward
builds it), the SDDMM (dc_edge_sddmm: K = 3 hop pairs for TAGConv, one pair + the self term for GCNConv) and the normalisation
backward (dc_gcn_norm_weighted_backward), each with its algorithmic bytes and their share of the 7.7 TB/s HBM bound.
Baseline, same process and inputs: the test reference (tests/edge_weight_reference.py) on stock PyTorch CUDA kernels, fp32,
TF32 off.  The working sets (x 524 MB, each hop 524 MB) exceed the 126 MB L2; no explicit flush between iterations.
Writes one JSON line per layer plus lines with the card, its power limit and SM clocks (query-only nvidia-smi).
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

HBM_BYTES_PER_S = 7.7e12


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


def norm_bytes(N, E, loops):
    """Algorithmic HBM bytes of dc_gcn_norm_weighted with both CSR orders: the two row-pointer arrays (8N), per edge and
    order the neighbour and edge id read, the weight gathered and the weight and record written (2 x 24E), the degree pass
    (edge ids and weights again, 8E) and dis (4N); with loops also edge_index (16E) and loop_w, loop_eid, self_w (12N)."""
    return 8 * N + 48 * E + 8 * E + 4 * N + ((16 * E + 12 * N) if loops else 0)


def norm_bwd_bytes(N, E, loops):
    """dc_gcn_norm_weighted_backward: both row-pointer arrays (8N), per edge and order neighbour, edge id, s and w (2 x 16E),
    the by-target pass again for dw (12E) and dw written (4E), dis (4N); with loops loop_w, loop_eid, s_self (12N)."""
    return 8 * N + 32 * E + 16 * E + 4 * N + (12 * N if loops else 0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSON-lines file to write")
    ap.add_argument("--graphs", type=int, default=256)
    ap.add_argument("--nodes", type=int, default=2000)
    ap.add_argument("--k", type=int, default=8)
    ap.add_argument("--fin", type=int, default=256)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--no-baseline", action="store_true", help="skip the reference baseline (fast rehearsal)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("edge_weight_bench.py measures on a CUDA device; none found")
    import deformcontact_b200 as dc
    from deformcontact_b200 import ops
    from edge_weight_reference import GCNConvWeighted, TAGConvWeighted

    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    info = gpu_info()
    B, n, k, F = args.graphs, args.nodes, args.k, args.fin
    N = B * n
    gen = torch.Generator(device=dev).manual_seed(0)
    pos = torch.rand(N, 3, generator=gen, device=dev) - 0.5
    ptr = torch.arange(B + 1, device=dev) * n
    ei = dc.knn_graph(pos, k, ptr=ptr)
    ptr = ptr.tolist()
    E = int(ei.shape[1])
    x = torch.randn(N, F, generator=gen, device=dev)
    w = torch.rand(E, generator=gen, device=dev) * 1.9 + 0.1
    gout = torch.randn(N, F, generator=gen, device=dev)
    it, wu = args.iters, args.warmup
    lines = [dict(kind="setup", workload=f"{B} kNN-{k} graphs x {n} nodes, N={N}, E={E}, F={F}", iters=it, warmup=wu,
                  timing="CUDA events around `iters` back-to-back calls after `warmup` calls", **info)]

    for name in ("TAGConv", "GCNConv"):
        torch.manual_seed(0)
        layer = getattr(dc, name)(F, F).to(dev)
        mode = "tag" if name == "TAGConv" else "gcn"
        xg = x.clone().requires_grad_(True)
        rec = dict(kind="layer", layer=f"{name}({F}, {F})")
        for case, ew in (("no_weights", None), ("weights_no_grad", w), ("weights_with_grad", w.clone().requires_grad_(True))):
            def fb():
                layer.zero_grad(set_to_none=True)
                xg.grad = None
                if ew is not None and ew.requires_grad:
                    ew.grad = None
                (layer(xg, ei, ew, ptr=ptr) if ew is not None else layer(xg, ei, ptr=ptr)).backward(gout)
            rec[f"fwd_bwd_ms_{case}"] = ev_time(fb, it, wu)
        rec["weights_overhead_no_grad"] = rec["fwd_bwd_ms_weights_no_grad"] / rec["fwd_bwd_ms_no_weights"]
        rec["weights_overhead_with_grad"] = rec["fwd_bwd_ms_weights_with_grad"] / rec["fwd_bwd_ms_no_weights"]

        # the new kernels one by one, on the layer's own intermediates
        g = ops.graph_csr(ei, N, mode, ptr)
        loops = mode == "gcn"
        kern, nbytes = {}, {}
        kern["dc_gcn_norm_weighted"] = ev_time(lambda: ops.weighted_view(g, w, True, 1.0, transpose=True), it, wu)
        nbytes["dc_gcn_norm_weighted"] = norm_bytes(N, E, loops)
        v = ops.weighted_view(g, w, True, 1.0, transpose=True)
        if name == "TAGConv":
            with torch.no_grad():
                xp = x.contiguous()
                _, hops = torch.ops.dcb200.tag_conv_weighted(xp, ei, w, [l.weight for l in layer.lins], layer.bias, False, True,
                                                             ops.GEMM_AUTO, ptr)
            K = layer.K
            hs = [xp] + [hops[:, i * F:(i + 1) * F] for i in range(K)]
            gs = [torch.randn(N, F, generator=gen, device=dev) for _ in range(K)]
            pairs, self_term = [(gs[i], hs[i]) for i in range(K)], False
        else:
            pairs, self_term = [(gout, torch.randn(N, F, generator=gen, device=dev))], True
        kern["dc_edge_sddmm"] = ev_time(lambda: ops.edge_sddmm(v, pairs, self_term), it, wu)
        nbytes["dc_edge_sddmm"] = ops.sddmm_bytes(N, E, F, len(pairs), self_term)
        s, s_self = ops.edge_sddmm(v, pairs, self_term)
        kern["dc_gcn_norm_weighted_backward"] = ev_time(lambda: ops.gcn_norm_backward(v, s, s_self), it, wu)
        nbytes["dc_gcn_norm_weighted_backward"] = norm_bwd_bytes(N, E, loops)
        rec["kernel_ms"] = kern
        rec["kernel_bytes"] = nbytes
        rec["kernel_hbm_share"] = {kk: nbytes[kk] / HBM_BYTES_PER_S / (kern[kk] * 1e-3) for kk in kern}
        del v, s, s_self, pairs

        if not args.no_baseline:
            ref = (TAGConvWeighted(F, F) if name == "TAGConv" else GCNConvWeighted(F, F)).to(dev)
            ref.load_state_dict(layer.state_dict())
            xr, wr = x.clone().requires_grad_(True), w.clone().requires_grad_(True)

            def fb_ref():
                ref.zero_grad(set_to_none=True)
                xr.grad = wr.grad = None
                ref(xr, ei, wr).backward(gout)
            rec["baseline_reference_fwd_bwd_ms_weights_with_grad"] = ev_time(fb_ref, it, wu)
            rec["speedup_vs_reference_weights_with_grad"] = (rec["baseline_reference_fwd_bwd_ms_weights_with_grad"]
                                                             / rec["fwd_bwd_ms_weights_with_grad"])
            with torch.no_grad():
                o_ref = ref(x, ei, w)
                rec["layer_vs_reference_rel_err"] = ((layer(x, ei, w, ptr=ptr) - o_ref).abs().max() / o_ref.abs().max()).item()
            del ref, xr, wr, o_ref
        del layer, xg
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
