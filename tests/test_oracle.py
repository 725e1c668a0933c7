"""CPU tests: the oracle against the reference-generated golden fixtures and against independent
formulations (dense fp64, scipy.sparse, cKDTree), plus property tests (SURVEY.md section 4 tier 1-3)."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch
from scipy.spatial import cKDTree

import oracle
from oracle import convs, synthetic
from helpers import assert_close, canonical


def _g(seed=0, n=200, e=1500):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n, 21, generator=g), torch.randint(0, n, (2, e), generator=g)


# ---------------------------------------------------------------- pinned against the reference's own code
def test_assemble_golden(golden_dir):
    """The oracle's mesh_to_graph / _feature_rigid / from_data_list restatement against the fixture produced by the
    reference's own utils/graph_utils.py:mesh_to_graph and loaders/common.py:_feature_rigid (make_golden_assemble.py)."""
    gold = torch.load(f"{golden_dir}/assemble.pt")
    soft = oracle.Batch.from_data_list([oracle.mesh_to_graph(v, t.long()) for v, t in gold["meshes"]])
    for k in ("x", "pos", "edge_index", "batch", "ptr"):
        assert torch.equal(getattr(soft, k), gold["soft"][k]), k
    sv, st = oracle.uv_sphere(0.05, 20)
    rigid = []
    for c, fv, f in zip(gold["centers"], gold["force_vec"], gold["force"]):
        d = oracle.mesh_to_graph(sv + c, st)
        n = d.x.shape[0]
        d.x = torch.cat([fv.repeat(n, 1), f.float().reshape(1).repeat(n, 1), d.x], dim=1)
        rigid.append(d)
    rb = oracle.Batch.from_data_list(rigid)
    for k in ("x", "pos", "edge_index", "batch", "ptr"):
        assert torch.equal(getattr(rb, k), gold["rigid"][k]), k


def test_posenc_golden(golden_dir):
    gold = torch.load(f"{golden_dir}/posenc.pt")
    assert torch.equal(oracle.to_log_freq(gold["pos"], 3, 1), gold["out"])


def test_gradient_consistency_loss_golden(golden_dir):
    gold = torch.load(f"{golden_dir}/gcl.pt")
    pred = oracle.Data(pos=gold["pred_pos"], edge_index=gold["edge_index"])
    rest = oracle.Data(pos=gold["rest_pos"], edge_index=gold["edge_index"])
    assert torch.equal(oracle.GradientConsistencyLoss()(pred, rest), gold["loss"])


@pytest.mark.parametrize("backbone", ["TAGConv", "GCNConv", "GATConv"])
def test_graphnet_wiring_golden(golden_dir, backbone):
    gold = torch.load(f"{golden_dir}/graphnet_{backbone}.pt")
    rest, rigid, _ = synthetic.make_batch(gold["n_graphs"], gold["n_nodes"], gold["k"])
    model = oracle.load_model(gold["kw"])
    model.load_state_dict(gold["state_dict"])
    out = model(rest, rigid)
    assert torch.equal(out.pos, gold["out_pos"])


def test_collate_golden(golden_dir):
    gold = torch.load(f"{golden_dir}/collate.pt")
    assert gold["n_rest"] == 3 and gold["meta_force_vector"].shape == (3, 3) and gold["meta_force"] == [0.0, 1.0, 2.0]


def test_self_pins(golden_dir):
    gold = torch.load(f"{golden_dir}/layers.pt")
    for name, rec in gold["layers"].items():
        layer = getattr(oracle, name)(21, 16)
        layer.load_state_dict(rec["state_dict"])
        assert torch.equal(layer(gold["x"], gold["edge_index"]), rec["out"])
    gg = torch.load(f"{golden_dir}/graphs.pt")
    assert torch.equal(oracle.knn_graph(gg["pts"], 5), gg["knn5"])
    assert torch.equal(oracle.knn_graph(gg["pts"], 5, gg["batch"]), gg["knn5_b"])
    assert torch.equal(oracle.radius_graph(gg["pts"], 0.15), gg["rad"])
    assert torch.equal(oracle.radius_graph(gg["pts"], 0.3, gg["batch"]), gg["rad_b"])


# ---------------------------------------------------------------- independent formulations
def test_tagconv_vs_dense_fp64_and_scipy():
    x, ei = _g()
    torch.manual_seed(0)
    layer = oracle.TAGConv(21, 32)
    with torch.no_grad():
        layer.bias.uniform_(-1, 1)
    out = layer(x, ei)
    ref = convs.tag_dense_fp64(x, ei, [l.weight for l in layer.lins], layer.bias)
    assert_close(out, ref.float(), what="TAGConv vs dense fp64")
    n = x.shape[0]
    A = sp.coo_matrix((np.ones(ei.shape[1]), (ei[1].numpy(), ei[0].numpy())), shape=(n, n)).tocsr()
    deg = np.asarray(A.sum(1)).ravel()
    dis = np.where(deg > 0, deg ** -0.5, 0.0)
    Ah = sp.diags(dis) @ A @ sp.diags(dis)
    h = x.double().numpy()
    acc = h @ layer.lins[0].weight.double().detach().numpy().T
    for lin in layer.lins[1:]:
        h = Ah @ h
        acc = acc + h @ lin.weight.double().detach().numpy().T
    assert_close(out, torch.from_numpy(acc + layer.bias.double().detach().numpy()).float(), what="TAGConv vs scipy")


def test_gcnconv_vs_dense():
    x, ei = _g(1)
    torch.manual_seed(1)
    layer = oracle.GCNConv(21, 16)
    n = x.shape[0]
    A = torch.zeros(n, n, dtype=torch.float64)
    m = ei[0] != ei[1]
    A.index_put_((ei[1][m], ei[0][m]), torch.ones(int(m.sum()), dtype=torch.float64), accumulate=True)
    A = A + torch.eye(n, dtype=torch.float64)
    dis = A.sum(1).pow(-0.5)
    ref = (dis[:, None] * A * dis[None, :]) @ (x.double() @ layer.lin.weight.double().t()) + layer.bias.double()
    assert_close(layer(x, ei), ref.float(), what="GCNConv vs dense")


def test_gatconv_vs_dense():
    x, ei = _g(2, n=60, e=400)
    ei = torch.unique(ei[:, ei[0] != ei[1]], dim=1)      # dense form cannot express duplicate edges
    torch.manual_seed(2)
    layer = oracle.GATConv(21, 8)
    xs = x.double() @ layer.lin.weight.double().t()
    a_s = (xs * layer.att_src.double().view(1, -1)).sum(-1)
    a_d = (xs * layer.att_dst.double().view(1, -1)).sum(-1)
    n = x.shape[0]
    mask = torch.eye(n, dtype=torch.bool)
    mask[ei[1], ei[0]] = True
    e = torch.nn.functional.leaky_relu(a_d[:, None] + a_s[None, :], 0.2).masked_fill(~mask, float("-inf"))
    ref = torch.softmax(e, dim=1) @ xs + layer.bias.double()
    assert_close(layer(x, ei), ref.float(), what="GATConv vs dense")


@pytest.mark.parametrize("name", ["TAGConv", "GCNConv", "GATConv"])
def test_properties(name):
    x, ei = _g(3)
    torch.manual_seed(3)
    layer = getattr(oracle, name)(21, 16)
    out = layer(x, ei)
    n = x.shape[0]
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(0))
    inv = torch.empty_like(perm)
    inv[perm] = torch.arange(n)
    assert_close(layer(x[perm], inv[ei]), out[perm], what="permutation equivariance")
    if name != "GATConv":   # linear in x (up to the bias)
        b = layer.bias
        assert_close(layer(2 * x, ei) - b, 2 * (out - b), what="linearity")
    # isolated node: TAG -> W0 x + b ; GCN/GAT -> its own (self-loop) transform
    ei2 = ei[:, (ei != 5).all(0)]
    o5 = layer(x, ei2)[5]
    if name == "TAGConv":
        assert_close(o5, layer.lins[0](x[5:6])[0] + layer.bias, what="isolated node")
    else:
        assert_close(o5, layer.lin(x[5:6])[0] + layer.bias, what="isolated node")
    # E = 0
    assert layer(x, torch.zeros(2, 0, dtype=torch.long)).shape == (n, 16)


def test_gcn_norm_weight_rounding():
    """H1: deg^-1/2 via pow(-0.5) then product: for k = 8, w = fl(fl(8^-.5)^2) = 0.12499999 != 0.125."""
    ei = torch.stack([torch.arange(1, 9), torch.zeros(8, dtype=torch.long)])
    ei = torch.cat([ei, torch.stack([torch.zeros(8, dtype=torch.long), torch.arange(1, 9)])], 1)
    ei = torch.cat([ei] + [torch.stack([torch.full((7,), i), torch.arange(1, 9)[torch.arange(1, 9) != i]]) for i in range(1, 9)], 1)
    _, w = convs.gcn_norm(ei, 9)
    d = torch.tensor(8.0).sqrt().reciprocal()
    assert (w == d * d).all()


# ---------------------------------------------------------------- kNN / radius vs KD-tree
def test_knn_vs_ckdtree():
    pts = torch.rand(700, 3, generator=torch.Generator().manual_seed(4))
    ei = oracle.knn_graph(pts, 6)
    _, idx = cKDTree(pts.double().numpy()).query(pts.double().numpy(), k=7)
    ref = {(int(j), i) for i in range(700) for j in idx[i][1:]}
    assert {(int(a), int(b)) for a, b in ei.t().tolist()} == ref
    assert ei.shape[1] == 700 * 6 and (ei[1] == torch.arange(700).repeat_interleave(6)).all()


def test_radius_vs_ckdtree():
    pts = torch.rand(500, 3, generator=torch.Generator().manual_seed(5))
    r = 0.12
    ei = oracle.radius_graph(pts, r, max_num_neighbors=64)
    pairs = cKDTree(pts.double().numpy()).query_pairs(r)
    got = {(min(a, b), max(a, b)) for a, b in ei.t().tolist()}
    # tie-free random input: fp32 vs fp64 threshold decisions agree except on measure-zero sets
    assert got == {(int(a), int(b)) for a, b in pairs}


def test_radius_truncation_rule():
    pts = torch.zeros(50, 3)
    pts[:, 0] = torch.arange(50) * 1e-3
    ei = oracle.radius_graph(pts, 1.0, max_num_neighbors=4)
    # query 0: first 5 by index incl. self -> {1,2,3,4}; query 40: first 5 = {0..4}, self absent -> 5 edges
    assert ei[0][ei[1] == 0].tolist() == [1, 2, 3, 4]
    assert ei[0][ei[1] == 40].tolist() == [0, 1, 2, 3, 4]


def test_knn_coincident_points_keep_k_plus_one():
    pts = torch.zeros(6, 3)
    ei = oracle.knn_graph(pts, 2)         # all distances tie at 0: top-3 by index = {0,1,2}
    assert ei[0][ei[1] == 5].tolist() == [0, 1, 2]          # self displaced -> k+1 edges
    assert ei[0][ei[1] == 1].tolist() == [0, 2]


def test_mesh_to_graph_order_and_sphere_counts():
    v, t = oracle.uv_sphere()
    assert v.shape == (762, 3) and t.shape == (1520, 3)
    d = oracle.mesh_to_graph(v, t)
    assert d.edge_index.shape == (2, 4560) and d.x.shape == (762, 21)
    a, b, c = t[0].tolist()
    assert d.edge_index[:, :3].t().tolist() == [[a, b], [b, c], [c, a]]
    s = set(map(tuple, d.edge_index.t().tolist()))
    assert all((q, p) in s for p, q in s)                    # closed, consistently oriented => symmetric


def test_batch_layout():
    rest, rigid, _ = synthetic.make_batch(3, 50, 4)
    assert rest.ptr.tolist() == [0, 50, 100, 150] and rest.batch.tolist() == sum(([g] * 50 for g in range(3)), [])
    assert (rest.edge_index[:, 200:400] >= 50).all() and (rest.edge_index[:, 200:400] < 100).all()
    g1 = rest[1]
    assert g1.edge_index.min() >= 0 and g1.edge_index.max() < 50 and g1.x.shape == (50, 21)
    assert canonical(g1.edge_index).shape == (2, 200)


def test_attn_group_equals_minibatches():
    """attn_group=G reproduces the reference run on mini-batches of G graphs."""
    rest, rigid, _ = synthetic.make_batch(4, 60, 4)
    torch.manual_seed(0)
    m = oracle.load_model(hidden_dim=16, attn_group=2)
    full = m(rest, rigid).pos
    m.attn_group = None
    parts = []
    for g0 in (0, 2):
        r = oracle.Batch.from_data_list([rest[g0], rest[g0 + 1]])
        g = oracle.Batch.from_data_list([rigid[g0], rigid[g0 + 1]])
        parts.append(m(r, g).pos)
    assert_close(full, torch.cat(parts), what="attn_group vs mini-batches")


@pytest.fixture
def fixture_threads():
    """train_loop.pt was written with 8 intra-op threads on an AVX-512 CPU.  How the fp32 products and reductions of the loop
    are split over threads decides their last bits, and Adam's first steps (m / sqrt(v)) turn a last-bit difference in a
    near-zero gradient into a weight difference above the elementwise bar of the test; with the same split the loop reproduces
    the fixture bit for bit on any such CPU, whatever its core count."""
    threads = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(threads)


def test_train_step_restatement_vs_reference_training_loop(golden_dir, fixture_threads):
    """The oracle's train step (oracle.train_step_loss + Adam, what every GPU train-step parity test compares against)
    reproduces the reference's OWN loop: train.py:train(config) executed unmodified for one epoch over three mini-batches
    (tests/golden/make_golden_train.py -> train_loop.pt): the three logged losses of every step, the validation loss
    (absolute positions, train.py:100-105) and the weights the loop saved."""
    from oracle import synthetic
    gold = torch.load(f"{golden_dir}/train_loop.pt")
    m = gold["meta"]

    def batch(first):
        rests, defs, rigids = [], [], []
        for g in range(first, first + m["batch"]):
            rest, deformed, gen = synthetic.soft_graph(g, m["nodes"], m["k"])
            ci = int(torch.randint(0, m["nodes"], (1,), generator=gen))
            rests.append(rest); defs.append(deformed); rigids.append(synthetic.rigid_graph(rest.pos[ci], gen))
        return tuple(oracle.Batch.from_data_list(l) for l in (rests, rigids, defs))

    torch.manual_seed(m["seed"])
    model = oracle.load_model(hidden_dim=m["hidden"])
    opt = torch.optim.Adam(model.parameters(), lr=m["lr"])
    model.train()
    for b, logged in enumerate(gold["steps"]):
        rest, rigid, deformed = batch(b * m["batch"])
        loss, l1, lc = oracle.train_step_loss(model, rest, rigid, deformed, lambda_gradient=m["lambda_gradient"])
        for got, key in ((loss, "tr_loss"), (l1, "tr_mse_loss"), (lc, "tr_consistency_loss")):
            assert abs(got.item() - logged[key]) <= 1e-6 * abs(logged[key]), (b, key, got.item(), logged[key])
        opt.zero_grad()
        loss.backward()
        opt.step()
    model.eval()
    with torch.no_grad():
        rest, rigid, deformed = batch(1000)
        pred = model(rest, rigid)
        val = torch.nn.functional.l1_loss(pred.pos, deformed.pos) + m["lambda_gradient"] * oracle.GradientConsistencyLoss()(pred, deformed)
    assert abs(val.item() - gold["validation_loss"]) <= 1e-6 * abs(gold["validation_loss"])
    sd = model.state_dict()
    assert set(sd) == set(gold["state_dict"])
    for k, v in gold["state_dict"].items():
        assert torch.allclose(sd[k], v, rtol=1e-6, atol=1e-8), k
