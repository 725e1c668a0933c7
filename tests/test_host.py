"""CPU tests of the host-side logic: C-ABI surface, batch layout, sharding, flat-gradient exchange."""
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_abi_exports_every_declared_symbol():
    """libdcb200.so loads and exports exactly the entry points include/dcb200.h declares."""
    from deformcontact_b200 import _abi
    hdr = open(os.path.join(ROOT, "include", "dcb200.h")).read()
    declared = set(re.findall(r"DC_API[^;(]*?\b(dc_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    lib = _abi.lib()
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in dcb200.h but not exported"
    assert declared == set(_abi.PROTOTYPES), (declared ^ set(_abi.PROTOTYPES))
    out = subprocess.run(["nm", "-D", "--defined-only", _abi.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (dc_[a-z0-9_]+)", out))
    assert exported == declared, exported ^ declared
    assert lib.dc_version() >= 100


def test_no_cpu_fallback():
    """The product path refuses CPU tensors instead of silently computing elsewhere."""
    import deformcontact_b200 as dc
    from deformcontact_b200 import _abi
    layer = dc.TAGConv(21, 8)
    with pytest.raises(_abi.DcError):
        layer(torch.randn(10, 21), torch.zeros(2, 0, dtype=torch.long))
    with pytest.raises(_abi.DcError):
        dc.knn_graph(torch.rand(10, 3), 3)


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "deformcontact_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f"{f} imports the oracle"


def test_state_dict_keys_match_pyg_names():
    import deformcontact_b200 as dc
    m = dc.load_model()
    keys = set(m.state_dict())
    for k in ("conv_layers_resting.0.lins.0.weight", "conv_layers_resting.1.lins.3.weight", "conv_layers_resting.0.bias",
              "conv_layers_rigid.1.lins.2.weight", "multihead_attention.attention_heads.1.weight", "decoder.0.weight",
              "decoder.9.bias"):
        assert k in keys, k
    assert sum(p.numel() for p in m.parameters()) == 1033219            # SURVEY.md 8(a) A1
    assert m.conv_layers_resting[0].lins[0].weight.shape == (256, 21)
    assert m.conv_layers_rigid[0].lins[0].weight.shape == (256, 25)
    g = dc.load_model(backbone="GATConv")
    assert {"conv_layers_resting.0.lin.weight", "conv_layers_resting.0.att_src", "conv_layers_resting.0.att_dst",
            "conv_layers_resting.0.bias"} <= set(g.state_dict())
    c = dc.load_model(backbone="GCNConv")
    assert {"conv_layers_rigid.0.lin.weight", "conv_layers_rigid.0.bias"} <= set(c.state_dict())


def test_load_model_from_reference_config_object():
    import deformcontact_b200 as dc

    class NS:
        pass
    cfg = NS()
    cfg.network = NS()
    for k, v in dc.EVERYDAY.items():
        setattr(cfg.network, k, v)
    m = dc.load_model(cfg)
    assert m.backbone == "TAGConv" and len(m.conv_layers_resting) == 2 and m.decoder[0].in_features == 768


def test_batch_layout_matches_oracle():
    import deformcontact_b200 as dc
    import oracle
    from oracle import synthetic
    rest, _, _ = synthetic.make_batch(3, 40, 4)
    mine = dc.Batch.from_data_list([dc.Data(x=d.x, edge_index=d.edge_index, pos=d.pos) for d in (rest[0], rest[1], rest[2])])
    for k in ("x", "pos", "edge_index", "batch", "ptr"):
        assert torch.equal(getattr(mine, k), getattr(rest, k)), k
    assert torch.equal(mine[2].edge_index, rest[2].edge_index)
    c = mine.clone()
    c.pos += 1
    assert not torch.equal(c.pos, mine.pos)


def test_collate_fn_matches_reference_semantics():
    import deformcontact_b200 as dc
    samples = [(f"o{i}", dc.Data(pos=torch.zeros(2, 3)), dc.Data(pos=torch.ones(2, 3)),
                {"force_vector": torch.full((3,), float(i)), "force": float(i), "path": f"p{i}"},
                dc.Data(pos=torch.zeros(1, 3))) for i in range(3)]
    names, rest, deformed, meta, rigid = dc.collate_fn(samples)
    assert names == ["o0", "o1", "o2"] and len(rest) == 3 and isinstance(rest, tuple)
    assert meta["force_vector"].shape == (3, 3) and meta["force"] == [0.0, 1.0, 2.0] and meta["path"] == ["p0", "p1", "p2"]


def test_shard_range():
    from deformcontact_b200 import dist
    for n, w in ((256, 8), (10, 4), (3, 8), (7, 1)):
        r = [dist.shard_range(n, i, w) for i in range(w)]
        assert r[0][0] == 0 and r[-1][1] == n and all(a[1] == b[0] for a, b in zip(r, r[1:]))
        sizes = [b - a for a, b in r]
        assert max(sizes) - min(sizes) <= 1
    r = [dist.shard_range(5, i, 2, [1, 1, 1, 10, 1]) for i in range(2)]
    assert r == [(0, 4), (4, 5)]


_WORKER = r'''
import os, sys, torch, torch.distributed as tdist
sys.path.insert(0, os.environ["DC_ROOT"])
from deformcontact_b200 import dist
rank, local, world = dist.init(backend="gloo")
torch.manual_seed(0)
net = torch.nn.Sequential(torch.nn.Linear(4, 3), torch.nn.Linear(3, 1))
flat = dist.FlatGrads(net.parameters())
g = torch.Generator().manual_seed(1)
X = torch.randn(12, 4, generator=g); Y = torch.randn(12, 1, generator=g)
sizes = [5, 7]                                    # unequal shards
lo = sum(sizes[:rank]); hi = lo + sizes[rank]
node_share, edge_share = dist.loss_shares(sizes[rank], sizes[rank], "cpu")
flat.zero_()
loss = node_share * torch.nn.functional.l1_loss(net(X[lo:hi]), Y[lo:hi])
loss.backward()
flat.all_reduce()
# reference: the global-mean loss on one process
ref = torch.nn.Sequential(torch.nn.Linear(4, 3), torch.nn.Linear(3, 1)); ref.load_state_dict(net.state_dict())
torch.nn.functional.l1_loss(ref(X), Y).backward()
refflat = torch.cat([p.grad.reshape(-1) for p in ref.parameters()])
assert torch.allclose(flat.flat, refflat, rtol=1e-5, atol=1e-7), (flat.flat, refflat)
assert all(p.grad.data_ptr() >= flat.flat.data_ptr() for p in net.parameters())
f, l = dist.shard_range(10, rank, world)
assert (f, l) == ((0, 5) if rank == 0 else (5, 10))
tdist.barrier(); tdist.destroy_process_group()
print("ok", rank)
'''


def test_flat_grad_allreduce_gloo_world2(tmp_path):
    """N>1 path on CPU: world_size-2 gloo; unequal shards reproduce the global-mean gradient."""
    import socket
    script = tmp_path / "w.py"
    script.write_text(_WORKER)
    with socket.socket() as s:      # a port nobody else on this host holds
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    env = dict(os.environ, DC_ROOT=ROOT, MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), WORLD_SIZE="2")
    procs = [subprocess.Popen([sys.executable, str(script)], env=dict(env, RANK=str(r), LOCAL_RANK=str(r)),
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=120)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o


def test_order_hints_are_weak_and_scoped():
    """ops.REORDER host logic: a hint lives as long as its edge_index tensor, is never pinned, and only one large
    TAG / GCN graph qualifies for relabelling."""
    import gc
    from deformcontact_b200 import ops
    n = ops.REORDER_MIN_NODES
    ei = torch.zeros((2, 7), dtype=torch.long)
    order = torch.arange(n, dtype=torch.int32)
    ops.register_order_hint(ei, order)
    assert ops._order_hint(ei, n) is order
    assert ops._order_hint(ei, n + 1) is None                              # node count must match
    assert ops._order_hint(torch.zeros((2, 7), dtype=torch.long), n) is None   # another tensor, another address
    assert ops._eligible_order(ei, n, "tag", None) is order
    assert ops._eligible_order(ei, n, "gcn", [0, n]) is order             # a single graph given as ptr
    assert ops._eligible_order(ei, n, "gat", None) is None                # GAT kernels read the CSR directly
    assert ops._eligible_order(ei, n, "tag", [0, 5, n]) is None           # block-diagonal batch: tiled by graph instead
    assert ops._eligible_order(ei, n - 1, "tag", None) is None            # small graph
    old, ops.REORDER = ops.REORDER, False
    try:
        assert ops._eligible_order(ei, n, "tag", None) is None
    finally:
        ops.REORDER = old
    key = ops._hint_key(ei)
    del ei
    gc.collect()
    assert ops._ORDER_HINTS[key][0]() is None                              # the table did not keep the tensor alive
    ops.register_order_hint(torch.zeros((2, 3), dtype=torch.long), order)  # registering prunes dead entries
    assert key not in ops._ORDER_HINTS


def test_tiles_are_closed_only_for_whole_graphs():
    """The hop chain (K1 v9) needs every tile to be closed under the edges: make_tiles merges small graphs and never
    splits one unless it exceeds the tile budget; the closure test is 'every tile boundary is a graph boundary'."""
    from deformcontact_b200 import ops
    ptr = [0, 762, 1524, 2286, 3048, 5048, 7048]                          # colliders (merged) + soft graphs
    tiles = ops.make_tiles(ptr, ptr[-1])
    assert tiles[0] == 0 and tiles[-1] == ptr[-1] and set(tiles) <= set(ptr)
    assert max(b - a for a, b in zip(tiles[:-1], tiles[1:])) <= ops.TILE_NODES + ops.TILE_NODES // 4
    big = [0, 3 * ops.TILE_NODES]                                          # one large graph is split -> not closed
    assert not set(ops.make_tiles(big, big[-1])) <= set(big)
    assert ops.make_tiles(None, 100) is None


def test_packer_layout_is_aligned_and_roundtrips():
    """assemble._Packer: typed arrays at 256-byte aligned offsets of one byte buffer; the same plan carves the device copy."""
    from deformcontact_b200 import assemble
    pk = assemble._Packer()
    pk.add("a", torch.int64, (3,))
    pk.add("b", torch.float32, (5, 3))
    pk.add("c", torch.int32, (2, 0))
    pk.add("d", torch.float64, (2, 3))
    assert all(off % 256 == 0 for _, _, _, off, _ in pk.fields) and pk.total % 256 == 0
    buf = torch.zeros(pk.total, dtype=torch.uint8)
    v = pk.views(buf)
    v["a"].copy_(torch.tensor([1, 2, 3]))
    v["b"].copy_(torch.arange(15.0).reshape(5, 3))
    v["d"].fill_(0.5)
    w = pk.views(buf.clone())
    assert w["a"].tolist() == [1, 2, 3] and torch.equal(w["b"], torch.arange(15.0).reshape(5, 3))
    assert w["c"].shape == (2, 0) and w["d"].dtype == torch.float64 and float(w["d"].sum()) == 3.0
    assert assemble._cumsum0([2, 0, 5]) == [0, 2, 2, 7]
    with pytest.raises(Exception):
        assemble.batch_from_data_list([], device="cuda")


@pytest.mark.parametrize("backbone", ["TAGConv", "GCNConv", "GATConv"])
def test_model_structure_matches_the_reference_loader(backbone):
    """A1: the reference's own Config(configs/everyday.json) + models/model_loader.py:load_model, executed unmodified
    (tests/golden/make_golden_loader.py -> loader.json): same network hyper-parameters, same state-dict keys and shapes,
    same parameter count and decoder layout for the product model and for the oracle — so reference checkpoints load."""
    import json
    import deformcontact_b200 as dc
    import oracle
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "loader.json")))[backbone]
    net = dict(gold["network"])
    assert {k: net[k] for k in dc.EVERYDAY if k != "backbone"} == {k: v for k, v in dc.EVERYDAY.items() if k != "backbone"}
    assert {k: v for k, v in oracle.EVERYDAY.items() if k != "backbone"} == {k: net[k] for k in oracle.EVERYDAY if k != "backbone"}

    class NS:
        pass
    cfg = NS()
    cfg.network = NS()
    for k, v in net.items():
        setattr(cfg.network, k, v)
    for model in (dc.load_model(cfg), oracle.load_model(backbone=backbone)):
        sd = {k: list(v.shape) for k, v in model.state_dict().items()}
        assert sd == gold["state_dict"]
        assert sum(p.numel() for p in model.parameters()) == gold["num_parameters"]
        assert [type(m).__name__ for m in model.decoder] == gold["decoder"]


def test_bench_strong_scaling_shards_one_batch():
    """bench.py --scaling strong (default): BASELINE C3 = ONE batch of 256 graphs split over the ranks; the per-rank ranges
    tile the batch exactly and the config says so on both arms."""
    import argparse
    import bench
    from deformcontact_b200 import dist
    for world in (1, 2, 4, 8):
        got = [dist.shard_range(256, r, world) for r in range(world)]
        assert got[0][0] == 0 and got[-1][1] == 256
        assert all(a[1] == b[0] for a, b in zip(got[:-1], got[1:]))
        assert all(hi - lo == 256 // world for lo, hi in got)
        args = argparse.Namespace(scaling="strong", global_batch=256, graphs_per_gpu=256, nodes=2000, k=8, attn_group=4)
        cfg = bench.config_dict(args, world)
        assert cfg["global_batch"] == 256 and cfg["graphs_per_gpu"] == 256 // world and cfg["parallelism"] == f"dp{world}"
    args = argparse.Namespace(scaling="weak", global_batch=256, graphs_per_gpu=64, nodes=2000, k=8, attn_group=4)
    assert bench.config_dict(args, 4)["global_batch"] == 256


def test_gemm_segment_chunks_cover_every_segment():
    """ops.gemm chains more than _abi.MAX_SEGS K-segments in groups (decoder fed by >= 4 attention heads, TAGConv K >= 4)."""
    from deformcontact_b200 import _abi
    for n in range(1, 12):
        groups = [list(range(n))[i:i + _abi.MAX_SEGS] for i in range(0, n, _abi.MAX_SEGS)]
        assert sum(groups, []) == list(range(n)) and all(1 <= len(g) <= _abi.MAX_SEGS for g in groups)


def test_narrow_tagconv_inputs_are_padded_to_one_chain_slice():
    """layers._pad4: widths that are not a multiple of 4 get zero columns up to the next multiple (16-byte rows); TAGConv inputs
    narrower than 32 (21 / 25 in configs/everyday.json) go to exactly 32 so that the layer's hops qualify for the chain kernel
    (F % 32 == 0).  The padding is exact zeros on both operands, so x W^T is unchanged."""
    from deformcontact_b200 import layers
    x = torch.randn(7, 21)
    ws = [torch.randn(5, 21) for _ in range(4)]
    xp, wp = layers._pad4(x, ws, chain=True)
    assert xp.shape == (7, 32) and all(w.shape == (5, 32) for w in wp)
    assert torch.equal(xp[:, :21], x) and not xp[:, 21:].any() and not wp[0][:, 21:].any()
    assert torch.allclose(xp @ wp[0].t(), x @ ws[0].t(), rtol=0, atol=1e-6)
    xp, wp = layers._pad4(x, ws)                       # the other layers: next multiple of 4
    assert xp.shape == (7, 24) and wp[0].shape == (5, 24)
    x64 = torch.randn(3, 64)
    assert layers._pad4(x64, ws, chain=True)[0] is x64  # nothing to do at hidden widths


def test_attention_groups_partition_the_batch():
    """attention._groups: consecutive groups of `attn_group` graphs (the reference's mini-batches); None = one group."""
    from deformcontact_b200 import attention
    ptr_s, ptr_r = [0, 10, 25, 25, 40, 60], [0, 3, 6, 9, 12, 15]
    g = attention._groups(ptr_s, ptr_r, 2)
    assert g == [(0, 25, 0, 6), (25, 40, 6, 12), (40, 60, 12, 15)]
    assert attention._groups(ptr_s, ptr_r, None) == [(0, 60, 0, 15)]
    assert sum(s1 - s0 for s0, s1, _, _ in g) == ptr_s[-1] and sum(r1 - r0 for _, _, r0, r1 in g) == ptr_r[-1]


def test_product_modules_have_no_undefined_names():
    """The product path cannot run here (no GPU, no CPU fallback), so a missing import would only surface on the GPU box:
    every name a function body loads must be bound in its module, its enclosing scopes or builtins (symtable walk)."""
    import builtins, glob, os, symtable
    root = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    files = glob.glob(os.path.join(root, "deformcontact_b200", "*.py")) + [os.path.join(root, "bench.py"), os.path.join(root, "__graft_entry__.py")]
    bad = []
    for f in files:
        top = symtable.symtable(open(f).read(), f, "exec")
        module_names = {s.get_name() for s in top.get_symbols() if s.is_assigned() or s.is_imported() or s.is_namespace()}

        def walk(tab):
            for s in tab.get_symbols():
                if s.is_global() and s.is_referenced() and not s.is_assigned():
                    n = s.get_name()
                    if n not in module_names and not hasattr(builtins, n) and n not in ("__file__", "__name__", "__doc__"):
                        bad.append((os.path.basename(f), tab.get_name(), n))
            for c in tab.get_children():
                walk(c)
        for c in top.get_children():
            walk(c)
        for s in top.get_symbols():   # module level: referenced but never bound
            n = s.get_name()
            if s.is_referenced() and not (s.is_assigned() or s.is_imported() or s.is_namespace()) and not hasattr(builtins, n) \
                    and n not in ("__file__", "__name__", "__doc__"):
                bad.append((os.path.basename(f), "<module>", n))
    assert not bad, bad


def test_batched_grid_cell_ranges_do_not_overlap():
    """K4g batched (csrc/knn_grid.cu): graph b owns the cells [base_b, base_b + cells_b) of one cell array with
    base_b = 2 * (ptr[b] // 8) + 66 * b in closed form (no prefix sum on the device).  A graph of n points uses at most
    2 * max(n // 8, 1) + 64 cells (grid_max_cells): the ranges must not overlap and must fit batched_total_cells — restated here
    because an overflow would be silent out-of-bounds counting."""
    import random
    rnd = random.Random(0)
    target = lambda n: max(n // 8, 1)
    max_cells = lambda n: 2 * target(n) + 64
    base = lambda first, b: 2 * (first // 8) + 66 * b
    total = lambda N, B: 2 * (N // 8) + 66 * B + 2
    for trial in range(2000):
        B = rnd.choice([2, 3, 7, 64, 500])
        sizes = [rnd.choice([0, 0, 1, 5, 7, 8, 9, 63, 64, 250, 2000, 5000, rnd.randrange(0, 40000)]) for _ in range(B)]
        ptr = [0]
        for n in sizes:
            ptr.append(ptr[-1] + n)
        for b in range(B):
            end = base(ptr[b], b) + max_cells(sizes[b])
            nxt = base(ptr[b + 1], b + 1) if b + 1 < B else total(ptr[-1], B)
            assert end <= nxt, (sizes, b)


def test_attention_group_matrices_are_row_blocks_of_one_matrix():
    """attention._group_matrices: groups of equal collider width share ONE [sum ns_g, nr] buffer (one softmax launch per head,
    rows 16-byte aligned for the TMA operands of the batched products); ragged widths fall back to one buffer per group."""
    from deformcontact_b200 import attention
    live = [(0, 300, 0, 762), (300, 500, 762, 1524), (500, 1100, 1524, 2286)]
    m = attention._group_matrices(live, "cpu")
    assert m.whole is not None and tuple(m.whole.shape) == (1100, 762) and m.whole.stride(0) == 764
    assert [tuple(b.shape) for b in m] == [(300, 762), (200, 762), (600, 762)]
    assert all(b.data_ptr() % 16 == 0 and b.stride(0) % 4 == 0 for b in m)
    assert m[1].data_ptr() == m.whole[300:].data_ptr() and m[2].data_ptr() == m.whole[500:].data_ptr()
    ragged = attention._group_matrices([(0, 10, 0, 5), (10, 30, 5, 12)], "cpu")
    assert ragged.whole is None and [tuple(b.shape) for b in ragged] == [(10, 5), (20, 7)]
    assert all(b.stride(0) % 4 == 0 for b in ragged)
