"""GPU (-m gpu): the CUDA path, called through the product API / C ABI, against the CPU oracle and
the golden vectors of the unmodified reference.  Tolerance: 1e-4 relative (BASELINE north_star),
measured against each tensor's max magnitude; index arrays are compared bit-exactly in
tests/test_host_logic.py."""
import os

import numpy as np
import pytest
import torch

from alignn_b200 import ops, synthetic
from alignn_b200.alignn import ALIGNN, ALIGNNConfig, EdgeGatedGraphConv
from alignn_b200.alignn_atomwise import EdgeGatedGraphConv as EdgeGatedGraphConvLN
from alignn_b200.graph import Graph
from oracle import alignn_oracle as O
from oracle import golden_inputs as GI
from tests.helpers import REL_TOL, assert_close, assert_dict_close, rel_err, to_oracle

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

CONV_TAGS = [("bn_train", "batchnorm", True), ("bn_eval", "batchnorm", False), ("ln", "layernorm", True)]


def _make_conv(norm, d, seed, train):
    conv = (EdgeGatedGraphConv if norm == "batchnorm" else EdgeGatedGraphConvLN)(d, d)
    GI.fill_state_dict(conv, seed)
    conv.train(train)
    return conv.to(DEV)


def _run_conv(conv, g, x, y, seed, d, need_edge_out=True):
    wx = GI.features(seed + 1, x.shape[0], d).to(DEV)
    wy = GI.features(seed + 2, y.shape[0], d).to(DEV)
    xi = x.to(DEV).clone().requires_grad_(True)
    yi = y.to(DEV).clone().requires_grad_(True)
    xo, yo = conv(g.to(DEV), xi, yi, _need_edge_out=need_edge_out)
    loss = (xo * wx).sum() + ((yo * wy).sum() if need_edge_out else 0.0)
    params = [p for p in conv.parameters()]
    grads = torch.autograd.grad(loss, [xi, yi] + params, allow_unused=True)
    out = {"x_out": xo, "y_out": yo, "gx": grads[0], "gy": grads[1]}
    for (n, p), gr in zip(conv.named_parameters(), grads[2:]):
        out["g." + n] = torch.zeros_like(p) if gr is None else gr
    if isinstance(conv.bn_nodes, torch.nn.BatchNorm1d):
        for bn in ("bn_nodes", "bn_edges"):
            out[f"{bn}.running_mean"] = getattr(conv, bn).running_mean
            out[f"{bn}.running_var"] = getattr(conv, bn).running_var
    return out


def _oracle_conv(norm, train, og, x, y, d, seed, need_edge_out=True, dtype=torch.float64):
    conv = O.EdgeGatedGraphConv(d, d, norm=norm).to(dtype)
    GI.fill_state_dict(conv, seed)
    conv.train(train)
    wx = GI.features(seed + 1, x.shape[0], d).to(dtype)
    wy = GI.features(seed + 2, y.shape[0], d).to(dtype)
    xi = x.to(dtype).clone().requires_grad_(True)
    yi = y.to(dtype).clone().requires_grad_(True)
    xo, yo = conv(og, xi, yi)
    loss = (xo * wx).sum() + ((yo * wy).sum() if need_edge_out else 0.0)
    grads = torch.autograd.grad(loss, [xi, yi] + list(conv.parameters()), allow_unused=True)
    out = {"x_out": xo, "y_out": yo, "gx": grads[0], "gy": grads[1]}
    for (n, p), gr in zip(conv.named_parameters(), grads[2:]):
        out["g." + n] = torch.zeros_like(p) if gr is None else gr
    if norm == "batchnorm":
        for bn in ("bn_nodes", "bn_edges"):
            out[f"{bn}.running_mean"] = getattr(conv, bn).running_mean
            out[f"{bn}.running_var"] = getattr(conv, bn).running_var
    return out


@pytest.mark.parametrize("tag,norm,train", CONV_TAGS)
def test_conv_jvasp_vs_reference_golden(golden_dir, tag, norm, train):
    """BASELINE config 1 (32 atoms, d=64) against the unmodified reference's outputs."""
    gold = np.load(os.path.join(golden_dir, "conv_jvasp_d64.npz"))
    jv = np.load(os.path.join(golden_dir, "jvasp_98225.npz"))
    g = Graph(jv["src"], jv["dst"], 32)
    x, y = GI.features(11, 32, 64), GI.features(12, g.num_edges(), 64)
    out = _run_conv(_make_conv(norm, 64, 100, train), g, x, y, 100, 64)
    ref = {k: gold[f"{tag}.{k}"] for k in out}
    assert_dict_close({k: GI.sample(v) for k, v in out.items()}, ref, what=tag)


@pytest.mark.parametrize("tag,norm,train", CONV_TAGS)
def test_conv_linegraph_d256_vs_reference_golden(golden_dir, tag, norm, train):
    gold = np.load(os.path.join(golden_dir, "conv_lg_d256.npz"))
    g, lg, _, _ = synthetic.make_batch(batch_size=1, atoms=10, k=12, seed=5)
    xm, z = GI.features(21, g.num_edges(), 256), GI.features(22, lg.num_edges(), 256)
    out = _run_conv(_make_conv(norm, 256, 200, train), lg, xm, z, 200, 256)
    for k in ("x_out", "y_out", "gx", "gy", "g.edge_gate.weight", "g.src_gate.bias", "g.bn_edges.weight",
              "g.bn_nodes.bias", "g.dst_update.weight"):
        assert_close(GI.sample(out[k]), gold[f"{tag}.{k}"], what=f"{tag}.{k}")


@pytest.mark.parametrize("norm,train", [("batchnorm", True), ("layernorm", True), ("batchnorm", False)])
@pytest.mark.parametrize("d", [32, 64, 128, 256])
def test_conv_all_widths_ragged_graph(norm, train, d):
    """Ragged k-NN multigraph (variable in-degree, multi-edges, self-image bonds), every supported d."""
    g, _, _, _ = synthetic.make_batch(batch_size=3, atoms=9, k=8, seed=d, regular=False, vary_atoms=True)
    x, y = GI.features(1, g.num_nodes(), d), GI.features(2, g.num_edges(), d)
    out = _run_conv(_make_conv(norm, d, 7, train), g, x, y, 7, d)
    ref = _oracle_conv(norm, train, to_oracle(g), x, y, d, 7)
    assert_dict_close(out, ref, what=f"{norm} d={d}")


def test_conv_dead_edge_output():
    """_need_edge_out=False (last ALIGNN layer's z, last GCN layer's y; SURVEY App. D-11)."""
    g, lg, _, _ = synthetic.make_batch(batch_size=2, atoms=6, k=6, seed=8)
    d = 64
    x, y = GI.features(1, lg.num_nodes(), d), GI.features(2, lg.num_edges(), d)
    for norm, train in (("batchnorm", True), ("layernorm", True)):
        out = _run_conv(_make_conv(norm, d, 9, train), lg, x, y, 9, d, need_edge_out=False)
        ref = _oracle_conv(norm, train, to_oracle(lg), x, y, d, 9, need_edge_out=False)
        assert out["y_out"] is None
        assert_dict_close(out, ref, what=f"dead {norm}", keys=[k for k in ref if k != "y_out"])


def test_conv_edge_cases_isolated_nodes_and_hubs():
    """In-degree 0 nodes (sum over no edges = 0, alignn.py:105-109) and a hub with 70 in-edges
    (more than one 32-edge chunk per warp)."""
    rng = np.random.default_rng(0)
    n = 12
    src = np.concatenate([rng.integers(0, n, 70), rng.integers(0, n, 20)])
    dst = np.concatenate([np.full(70, 3), rng.integers(4, 8, 20)])      # nodes 0-2, 8-11 have no in-edges
    g = Graph(src, dst, n)
    d = 64
    x, y = GI.features(3, n, d), GI.features(4, g.num_edges(), d)
    for norm in ("batchnorm", "layernorm"):
        out = _run_conv(_make_conv(norm, d, 5, True), g, x, y, 5, d)
        ref = _oracle_conv(norm, True, to_oracle(g), x, y, d, 5)
        assert_dict_close(out, ref, what=f"edge-case {norm}")


def test_gather_segment_sum_primitive():
    """BASELINE config 5 primitive at 1e5 edges vs index_add; plus linearity at full size."""
    g, bh, sigma = synthetic.make_segment_sweep(100_000, d=256)
    gd = g.to(DEV)
    Sh, S = ops.gather_segment_sum(gd.index, bh.to(DEV), sigma.to(DEV))
    s, d = g.edges()
    ref_Sh = torch.zeros_like(bh, dtype=torch.float64).index_add(0, d.long(), (bh[s.long()] * sigma).double())
    ref_S = torch.zeros_like(bh, dtype=torch.float64).index_add(0, d.long(), sigma.double())
    assert_close(Sh, ref_Sh, tol=1e-5, what="Sh")
    assert_close(S, ref_S, tol=1e-5, what="S")
    # size-independent property: Sh is linear in Bh, S does not depend on Bh
    Sh2, S2 = ops.gather_segment_sum(gd.index, 2 * bh.to(DEV), sigma.to(DEV))
    assert torch.equal(Sh2, 2 * Sh) and torch.equal(S2, S)


SMALL_CFG = dict(alignn_layers=2, gcn_layers=2, hidden_features=64, embedding_features=32)
GRAD_KEYS = ("fc.weight", "atom_embedding.layer.0.weight", "alignn_layers.0.edge_update.edge_gate.weight",
             "alignn_layers.1.node_update.src_gate.weight", "gcn_layers.1.dst_update.bias",
             "alignn_layers.0.node_update.bn_nodes.weight", "gcn_layers.0.bn_edges.bias",
             "angle_embedding.1.layer.0.weight")


@pytest.mark.parametrize("case", ["reg", "knn"])
@pytest.mark.parametrize("train", [True, False])
def test_full_alignn_vs_reference_golden(golden_dir, case, train):
    gold = np.load(os.path.join(golden_dir, "alignn_small.npz"))
    if case == "reg":
        g, lg, lat, tgt = synthetic.make_batch(batch_size=3, atoms=9, k=12, seed=31, vary_atoms=True)
    else:
        g, lg, lat, tgt = synthetic.make_batch(batch_size=2, atoms=6, k=6, seed=32, regular=False)
    m = ALIGNN(ALIGNNConfig(name="alignn", **SMALL_CFG))
    GI.fill_state_dict(m, 300)
    m.to(DEV).train(train)
    out = m((g.to(DEV), lg.to(DEV), lat.to(DEV)))
    loss = (out - tgt.to(DEV)).abs().mean()
    loss.backward()
    tag = f"{case}.{'train' if train else 'eval'}"
    assert_close(out, gold[tag + ".out"], what="out")
    grads = dict(m.named_parameters())
    for k in GRAD_KEYS:
        gr = grads[k].grad
        got = torch.zeros_like(grads[k]) if gr is None else gr
        ref = gold[f"{tag}.g.{k}"]
        if np.abs(ref).max() == 0:
            assert float(got.abs().max()) == 0.0, k       # unused parameters (App. D-11) get no gradient
        else:
            assert_close(got, ref, tol=REL_TOL, what=k)


def _full_size_models(norm):
    if norm == "layernorm":
        from alignn_b200 import alignn_atomwise as AW

        class Model(ALIGNN):
            _mlp, _alignn_conv, _gcn_conv = AW.MLPLayer, AW.ALIGNNConv, AW.EdgeGatedGraphConv
        m = Model(ALIGNNConfig(name="alignn"))
    else:
        m = ALIGNN(ALIGNNConfig(name="alignn"))
    GI.fill_state_dict(m, 1234)
    orc = O.ALIGNN(norm=norm).double()
    orc.load_state_dict({k: v.double() if v.is_floating_point() else v for k, v in m.state_dict().items()})
    return m.to(DEV), orc


@pytest.mark.parametrize("norm", ["batchnorm", "layernorm"])
def test_full_size_batch64_vs_fp64_oracle(norm):
    """BASELINE configs 2/3 at full size (B=64, n=30, k=12, 4+4 layers, d=256, T = 276 480 bond pairs): inference
    output, training output and EVERY parameter gradient against the fp64 CPU oracle, tolerance 1e-4 of each tensor's
    scale (north_star).  Gradients that are mathematically zero (a bias feeding a train-mode BatchNorm, the dead norm
    layers of SURVEY App. D-11) are judged against the scale of their layer's other gradients."""
    g, lg, lat, tgt = synthetic.make_batch(batch_size=64, atoms=30, k=12, seed=123)
    m, orc = _full_size_models(norm)
    gd, lgd, latd = g.to(DEV), lg.to(DEV), lat.to(DEV)
    og, olg = to_oracle(g, torch.float64), to_oracle(lg, torch.float64)
    m.eval()
    orc.eval()
    with torch.no_grad():
        out = m((gd, lgd, latd))
        ref = orc((og, olg, lat))
    assert_close(out, ref, what=f"batch-64 {norm} inference")
    m.train()
    orc.train()
    out = m((gd, lgd, latd))
    (out - tgt.to(DEV)).abs().mean().backward()
    ref = orc((og, olg, lat))
    (ref - tgt.double()).abs().mean().backward()
    assert_close(out, ref, what=f"batch-64 {norm} train forward")
    got = {"g." + n: (p.grad if p.grad is not None else torch.zeros_like(p)) for n, p in m.named_parameters()}
    want = {"g." + n: (p.grad if p.grad is not None else torch.zeros_like(p)) for n, p in orc.named_parameters()}
    assert set(got) == set(want)
    assert_dict_close(got, want, what=f"batch-64 {norm}")
    if norm == "batchnorm":      # running statistics of every BatchNorm, dead ones included (App. D-11)
        bufs = dict(orc.named_buffers())
        for n, b in m.named_buffers():
            if n.endswith("running_mean") or n.endswith("running_var"):
                assert_close(b, bufs[n], what=n)


def test_cuda_graph_replay_and_host_batches_bit_identical_to_eager():
    """What bench.py times (CUDA-graph replay of forward+backward, batches copied from pinned host memory) produces
    bit-identical losses and gradients to plain eager launches on resident batches."""
    g, lg, lat, tgt = synthetic.make_batch(batch_size=8, atoms=12, k=12, seed=7)
    m = ALIGNN(ALIGNNConfig(name="alignn", alignn_layers=2, gcn_layers=2, hidden_features=64, embedding_features=32))
    GI.fill_state_dict(m, 5)
    m.to(DEV).train()
    host = (g.pin_memory(), lg.pin_memory(), lat.pin_memory(), tgt.pin_memory())

    def fwd_bwd(batch):
        gg, ll, la, tt = batch
        for p in m.parameters():
            p.grad = None
        loss = (m((gg, ll, la)) - tt).abs().mean()
        loss.backward()
        return loss

    def snapshot():
        return {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None}

    def reset_bn():
        for mod in m.modules():
            if isinstance(mod, torch.nn.BatchNorm1d):
                mod.reset_running_stats()
    res = tuple(t.to(DEV) for t in host)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            fwd_bwd(res)
    torch.cuda.current_stream().wait_stream(side)
    reset_bn()
    loss_eager = fwd_bwd(res).item()
    grads_eager = snapshot()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        loss_g = fwd_bwd(tuple(t.to(DEV, non_blocking=True) for t in host))
    for _ in range(2):
        gr.replay()
    torch.cuda.synchronize()
    assert loss_g.item() == loss_eager
    grads_graph = snapshot()
    assert set(grads_graph) == set(grads_eager)
    for n in grads_eager:
        assert torch.equal(grads_eager[n], grads_graph[n]), n


def test_force_training_on_gpu_matches_oracle_double_backward():
    """ALIGNN-FF training step with a force loss (create_graph=True through the conv stack, alignn_atomwise.py:530-539):
    on the GPU the convs run as torch-operator compositions (conv.second_order); parameter gradients against the fp64
    oracle's double backward."""
    from alignn_b200.alignn_atomwise import ALIGNNAtomWise, ALIGNNAtomWiseConfig
    g, lg, lat, _ = synthetic.make_batch(batch_size=2, atoms=8, k=12, seed=41, vary_atoms=True)
    m = ALIGNNAtomWise(ALIGNNAtomWiseConfig(name="alignn_atomwise", alignn_layers=2, gcn_layers=2, hidden_features=64,
                                            embedding_features=32, atom_input_features=92))
    GI.fill_state_dict(m, 400)
    orc = O.ALIGNN(norm="layernorm", alignn_layers=2, gcn_layers=2, hidden_features=64, embedding_features=32).double().train()
    orc.load_state_dict({k: v.double() for k, v in m.state_dict().items()})
    m.to(DEV).train()
    tgt_f = GI.features(12, g.num_nodes(), 3)
    res = m((g.to(DEV), lg.to(DEV), lat.to(DEV)))
    assert res["grad"].requires_grad
    ((res["grad"] - tgt_f.to(DEV)).abs().mean() + res["out"].abs().mean()).backward()
    out, forces, _ = O.energy_and_forces(orc, to_oracle(g, torch.float64), to_oracle(lg, torch.float64), create_graph=True)
    ((forces - tgt_f.double()).abs().mean() + out.abs().mean()).backward()
    got = {"g." + n: (p.grad if p.grad is not None else torch.zeros_like(p)) for n, p in m.named_parameters()}
    want = {"g." + n: (p.grad if p.grad is not None else torch.zeros_like(p)) for n, p in orc.named_parameters()}
    assert_dict_close(got, want, tol=1e-3, what="force-training gradients (fp32 ATen double backward vs fp64)")
    # and the same model serves inference / MD through the CUDA kernels
    m.eval()
    res_eval = m((g.to(DEV), lg.to(DEV), lat.to(DEV)))
    assert not res_eval["grad"].requires_grad
    assert_close(res_eval["grad"], forces.detach(), what="forces, kernel path vs oracle")


def test_deterministic_and_graph_not_mutated():
    g, lg, lat, tgt = synthetic.make_batch(batch_size=4, atoms=10, k=12, seed=77)
    m = ALIGNN(ALIGNNConfig(name="alignn", **SMALL_CFG)).to(DEV).train()
    gd, lgd = g.to(DEV), lg.to(DEV)
    keys = (set(gd.ndata), set(gd.edata), set(lgd.ndata), set(lgd.edata))
    outs, grads = [], []
    for _ in range(2):
        m.zero_grad()
        out = m((gd, lgd, lat.to(DEV)))
        out.sum().backward()
        outs.append(out.detach().clone())
        grads.append(m.alignn_layers[0].edge_update.edge_gate.weight.grad.clone())
    assert torch.equal(outs[0], outs[1]) and torch.equal(grads[0], grads[1])       # no float atomics anywhere
    assert keys == (set(gd.ndata), set(gd.edata), set(lgd.ndata), set(lgd.edata))   # inputs are borrowed


def test_launch_counter_counts_library_kernels():
    from alignn_b200 import _lib
    g, _, _, _ = synthetic.make_batch(batch_size=1, atoms=6, k=6, seed=2)
    conv = _make_conv("layernorm", 64, 3, True)
    before = _lib.launch_count()
    with torch.no_grad():
        conv(g.to(DEV), GI.features(1, g.num_nodes(), 64).to(DEV), GI.features(2, g.num_edges(), 64).to(DEV))
    # 2 table-driven refresh launches (operand images, bias vectors: once per weight change, not per call) +
    # node-projection GEMM + gather GEMM (gate) + segment-reduce kernel
    assert _lib.launch_count() - before == 5
    before = _lib.launch_count()
    with torch.no_grad():
        conv(g.to(DEV), GI.features(1, g.num_nodes(), 64).to(DEV), GI.features(2, g.num_edges(), 64).to(DEV))
    assert _lib.launch_count() - before == 3      # weights unchanged: no refresh


def test_atomwise_energy_and_forces_vs_reference_golden(golden_dir):
    """BASELINE config 4 path (ALIGNN-FF energy + forces by autograd through the conv stack) against the
    unmodified reference's ALIGNNAtomWise outputs."""
    from alignn_b200.alignn_atomwise import ALIGNNAtomWise, ALIGNNAtomWiseConfig
    gold = np.load(os.path.join(golden_dir, "atomwise_small.npz"))
    g, lg, lat, _ = synthetic.make_batch(batch_size=2, atoms=8, k=12, seed=41, vary_atoms=True)
    m = ALIGNNAtomWise(ALIGNNAtomWiseConfig(name="alignn_atomwise", alignn_layers=2, gcn_layers=2, hidden_features=64,
                                            embedding_features=32, atom_input_features=92))
    GI.fill_state_dict(m, 400)
    m.to(DEV).eval()
    res = m((g.to(DEV), lg.to(DEV), lat.to(DEV)))
    assert_close(res["out"], gold["out"], what="energy per atom")
    assert_close(res["grad"], gold["forces"], what="forces")
    assert_close(res["pair_forces"], gold["pair_forces"], what="pair forces")
    # size-independent property (test_force_reduction.py:212-229): net force on every crystal is zero
    off = g.node_graph_offsets().tolist()
    for a, b in zip(off[:-1], off[1:]):
        assert float(res["grad"][a:b].sum(0).abs().max()) < 1e-4


def test_edgeless_graph_and_single_node():
    """Empty edge set (isolated atoms): sums over no edges are 0 (alignn.py:105-109); nothing may read out of bounds."""
    g = Graph(np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.int64), 5)
    d = 64
    x, y = GI.features(1, 5, d), torch.zeros(0, d)
    for norm in ("layernorm", "batchnorm"):
        conv = _make_conv(norm, d, 11, True)
        xi = x.to(DEV).requires_grad_(True)
        xo, yo = conv(g.to(DEV), xi, y.to(DEV))
        xo.sum().backward()
        oc = O.EdgeGatedGraphConv(d, d, norm=norm).double()
        GI.fill_state_dict(oc, 11)
        xr = x.double().requires_grad_(True)
        xo_ref, _ = oc(to_oracle(g), xr, y.double())
        xo_ref.sum().backward()
        assert yo.shape == (0, d)
        assert_close(xo, xo_ref, what=f"edgeless {norm} x_out")
        assert_close(xi.grad, xr.grad, what=f"edgeless {norm} gx", atol=1e-5)



def test_atomwise_stress_vs_reference_golden(golden_dir):
    """Stress head of ALIGNN-FF (alignn_atomwise.py:567-638, batch_stress=True) through the CUDA conv stack against
    the unmodified reference's `result["stresses"]`."""
    from alignn_b200.alignn_atomwise import ALIGNNAtomWise, ALIGNNAtomWiseConfig
    gold = np.load(os.path.join(golden_dir, "atomwise_stress.npz"))
    g, lg, lat, _ = synthetic.make_batch(batch_size=2, atoms=8, k=12, seed=41, vary_atoms=True)
    g.ndata["V"] = GI.cell_volumes(g.batch_num_nodes())
    m = ALIGNNAtomWise(ALIGNNAtomWiseConfig(name="alignn_atomwise", alignn_layers=2, gcn_layers=2, hidden_features=64,
                                            embedding_features=32, atom_input_features=92, stresswise_weight=0.1,
                                            stress_multiplier=10.0))
    GI.fill_state_dict(m, 400)
    m.to(DEV).eval()
    res = m((g.to(DEV), lg.to(DEV), lat.to(DEV)))
    assert res["stresses"].shape == (2, 3, 3)
    # (1) the tail itself: fp64 loop restatement (oracle) applied to the pair forces this very run produced
    og = to_oracle(g, torch.float64)
    tail = O.virial_stress(og, res["pair_forces"].double().cpu(), g.ndata["V"].double(), stress_multiplier=10.0)
    assert_close(res["stresses"], tail, tol=1e-5, what="stress tail vs oracle on the same pair forces")
    # (2) end to end against the reference.  Each entry is a signed sum over ~100 bonds of r (up to 8 A) x pair force,
    # so the 1e-4 per-bond tolerance of the pair forces (checked above) propagates to ~1e-3 of the largest component.
    assert_close(res["stresses"], gold["stresses"], tol=1e-3, what="stress vs reference")


@pytest.mark.parametrize("tag", ["mult", "repl", "leak"])
def test_atomwise_cutoff_and_penalty_variants_vs_reference_golden(golden_dir, tag):
    """ALIGNN-FF with the cutoff envelope (both `multiply_cutoff` settings) and with the penalty leaking into `out`
    (energy_mult_natoms=False) against the unmodified reference; bonds shortened to 0.5-2.8 A as in the fixture."""
    from alignn_b200.alignn_atomwise import ALIGNNAtomWise, ALIGNNAtomWiseConfig
    cases = {"mult": dict(use_cutoff_function=True, multiply_cutoff=True, inner_cutoff=2.5, exponent=5),
             "repl": dict(use_cutoff_function=True, multiply_cutoff=False, inner_cutoff=2.5, exponent=3),
             "leak": dict(use_cutoff_function=False, penalty_threshold=1.2)}
    gold = np.load(os.path.join(golden_dir, "atomwise_cutoff.npz"))
    g, lg, lat, _ = synthetic.make_batch(batch_size=2, atoms=8, k=12, seed=41, vary_atoms=True)
    g.edata["r"] = g.edata["r"] * 0.35
    m = ALIGNNAtomWise(ALIGNNAtomWiseConfig(name="alignn_atomwise", alignn_layers=2, gcn_layers=2, hidden_features=64,
                                            embedding_features=32, atom_input_features=92,
                                            energy_mult_natoms=tag != "leak", **cases[tag]))
    GI.fill_state_dict(m, 400)
    m.to(DEV).eval()
    res = m((g.to(DEV), lg.to(DEV), lat.to(DEV)))
    assert_close(res["out"], gold[tag + ".out"], what=f"{tag} energy")
    assert_close(res["grad"], gold[tag + ".forces"], what=f"{tag} forces")


def test_config4_supercell_1000_atoms_energy_and_forces_vs_fp64_oracle():
    """BASELINE config 4 at full size: ALIGNN-FF (4+4 layers, d=256, LayerNorm) energy + per-atom forces on a 1000-atom
    periodic diamond supercell (radius graph 4 A, thermal jitter), structure built ON THE DEVICE, against the fp64
    oracle on the oracle's own restatement of the same neighbour list."""
    from alignn_b200 import neighbors
    from alignn_b200.alignn_atomwise import ALIGNNAtomWise, ALIGNNAtomWiseConfig
    lat, X = neighbors.diamond_supercell(reps=5, jitter=0.03, seed=1)
    feats = GI.features(5, X.shape[0], 92)
    g, lg = neighbors.crystal_graph_device(lat, X, feats, cutoff=4.0, device=DEV)
    # the oracle builds its own graph (restatement of alignn/graphs.py:267-364); both must agree bond for bond
    ou, ov, orr = O.radius_graph(lat, X, cutoff=4.0)[:3]
    assert g.num_nodes() == 1000 and g.num_edges() == len(ou)           # whatever the jitter makes of the 16-neighbour shell
    s, d = g.edges()
    assert np.array_equal(s.cpu().numpy(), np.asarray(ou)) and np.array_equal(d.cpu().numpy(), np.asarray(ov))
    og = O.OGraph(ou, ov, 1000)
    og.ndata["atom_features"] = feats.double()
    og.edata["r"] = torch.as_tensor(np.asarray(orr), dtype=torch.float64)
    olg = O.line_graph(og)
    m = ALIGNNAtomWise(ALIGNNAtomWiseConfig(name="alignn_atomwise", atom_input_features=92, alignn_layers=4, gcn_layers=4,
                                            hidden_features=256))
    GI.fill_state_dict(m, 900)
    orc = O.ALIGNN(norm="layernorm").double().eval()
    orc.load_state_dict({k: v.double() for k, v in m.state_dict().items()})
    m.to(DEV).eval()
    latd = torch.from_numpy(lat).float().unsqueeze(0).to(DEV)
    res = m((g, lg, latd))
    out, forces, pair = O.energy_and_forces(orc, og, olg)
    assert_close(res["out"], out, what="supercell energy per atom")
    assert_close(res["pair_forces"], pair, what="supercell pair forces")
    assert_close(res["grad"], forces, what="supercell forces")
    assert float(res["grad"].sum(0).abs().max()) < 1e-3 * float(res["grad"].abs().max()) * 1000 ** 0.5   # net force ~ 0


def test_force_reduction_properties_on_the_cuda_path():
    """The reference's two property tests for this path (alignn/tests/test_force_reduction.py:212-271) on the CUDA
    kernels: (1) Newton's third law -- the forces of every crystal sum to zero; (2) the in-edge / out-edge reduction of
    the pair forces equals the force assembled bond by bond (what the reference compares against position gradients)."""
    from alignn_b200.alignn_atomwise import ALIGNNAtomWise, ALIGNNAtomWiseConfig
    g, lg, lat, _ = synthetic.make_batch(batch_size=3, atoms=10, k=12, seed=43, vary_atoms=True)
    m = ALIGNNAtomWise(ALIGNNAtomWiseConfig(name="alignn_atomwise", alignn_layers=2, gcn_layers=2, hidden_features=64,
                                            embedding_features=32, atom_input_features=92))
    GI.fill_state_dict(m, 401)
    m.to(DEV).eval()
    res = m((g.to(DEV), lg.to(DEV), lat.to(DEV)))
    f, pf = res["grad"].double().cpu(), res["pair_forces"].double().cpu()
    off = g.node_graph_offsets().tolist()
    scale = float(f.abs().max())
    for a, b in zip(off[:-1], off[1:]):
        assert float(f[a:b].sum(0).abs().max()) <= 1e-5 * scale * (b - a)
    s, d = (t.long() for t in g.edges())
    by_bond = torch.zeros_like(f)
    for e in range(g.num_edges()):                      # plain loop: +F on the destination atom, -F on the source atom
        by_bond[d[e]] += pf[e]
        by_bond[s[e]] -= pf[e]
    assert float((f - by_bond).abs().max()) <= 1e-5 * scale


def test_bn_links_move_the_batchnorm_backward_reductions_into_the_gemm_epilogue():
    """(Optional path, off by default: measured slower, see ops.USE_BN_LINKS.)  With ops.BNLink the T-sized reductions of the train-mode BatchNorm backward (one per L(g) conv that has a
    consumer, plus the angle embedding's last layer) ride on the consumer's data-gradient GEMM; results equal the
    explicit reduction pass to fp32 round-off."""
    g, lg, lat, tgt = synthetic.make_batch(batch_size=4, atoms=10, k=12, seed=9)
    gd, lgd, latd, tgtd = g.to(DEV), lg.to(DEV), lat.to(DEV), tgt.to(DEV)

    def run(use_links):
        ops.USE_BN_LINKS = use_links
        m = ALIGNN(ALIGNNConfig(name="alignn", alignn_layers=3, gcn_layers=1, hidden_features=64, embedding_features=32))
        GI.fill_state_dict(m, 21)
        m.to(DEV).train()
        ops.TIMER = ops.KernelTimer()
        (m((gd, lgd, latd)) - tgtd).abs().mean().backward()
        torch.cuda.synchronize()
        names = {k: len(v) for k, v in ops.TIMER.records.items()}
        ops.TIMER = None
        return {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None}, names
    try:
        g_on, n_on = run(True)
        g_off, n_off = run(False)
    finally:
        ops.USE_BN_LINKS = False
        ops.TIMER = None
    fused = sum(v for k, v in n_on.items() if "bn_bwd" in k)
    assert fused >= 3                                   # L(g) convs 1, 2 -> 0, 1 and layer 0 -> angle embedding (+ g-side links)
    assert n_on.get("bn_backward_reduce", 0) <= n_off["bn_backward_reduce"] - fused
    for k in g_off:
        scale = max(g_off[k].abs().max().item(), 1e-12)
        assert (g_on[k] - g_off[k]).abs().max().item() <= 2e-5 * scale + 1e-7, k
