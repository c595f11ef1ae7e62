"""CPU: the oracle restatement vs golden vectors produced by the UNMODIFIED reference
(oracle/make_golden.py).  Also the reference's own property tests for this path
(alignn/tests/test_force_reduction.py:212-271) restated on the oracle."""
import os

import numpy as np
import pytest
import torch

from alignn_b200 import synthetic
from oracle import alignn_oracle as O
from oracle import golden_inputs as GI
from tests.helpers import to_oracle


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


def _conv_run(norm, train, og, x, y, d, seed, dtype):
    conv = O.EdgeGatedGraphConv(d, d, norm=norm).to(dtype)
    GI.fill_state_dict(conv, seed)
    conv.train(train)
    wx = GI.features(seed + 1, x.shape[0], d).to(dtype)
    wy = GI.features(seed + 2, y.shape[0], d).to(dtype)
    xi = x.to(dtype).clone().requires_grad_(True)
    yi = y.to(dtype).clone().requires_grad_(True)
    xo, yo = conv(og, xi, yi)
    loss = (xo * wx).sum() + (yo * wy).sum()
    grads = torch.autograd.grad(loss, [xi, yi] + list(conv.parameters()))
    out = {"x_out": xo, "y_out": yo, "gx": grads[0], "gy": grads[1]}
    for (n, _), g in zip(conv.named_parameters(), grads[2:]):
        out["g." + n] = g
    if norm == "batchnorm":
        for bn in ("bn_nodes", "bn_edges"):
            out[f"{bn}.running_mean"] = getattr(conv, bn).running_mean
            out[f"{bn}.running_var"] = getattr(conv, bn).running_var
    return out


CONV_TAGS = [("bn_train", "batchnorm", True), ("bn_eval", "batchnorm", False), ("ln", "layernorm", True)]


@pytest.mark.parametrize("tag,norm,train", CONV_TAGS)
def test_conv_jvasp_matches_reference_fp64(golden_dir, tag, norm, train):
    """BASELINE config 1 shape: one EdgeGatedGraphConv on the 32-atom JVASP-98225 radius graph, d=64."""
    gold = _load(golden_dir, "conv_jvasp_d64.npz")
    jv = _load(golden_dir, "jvasp_98225.npz")
    s, d_ = torch.from_numpy(jv["src"]), torch.from_numpy(jv["dst"])
    x, y = GI.features(11, 32, 64), GI.features(12, s.numel(), 64)
    assert GI.checksum(x, y, s, d_) == int(gold["in_crc"]), "seeded inputs drifted from the fixture"
    out = _conv_run(norm, train, O.OGraph(s, d_, 32), x, y, 64, 100, torch.float64)
    for k, v in out.items():
        ref = gold[f"{tag}.{k}"]
        np.testing.assert_allclose(GI.sample(v), ref, rtol=1e-10, atol=1e-11, err_msg=f"{tag}.{k}")


@pytest.mark.parametrize("tag,norm,train", CONV_TAGS)
def test_conv_linegraph_d256_matches_reference(golden_dir, tag, norm, train):
    gold = _load(golden_dir, "conv_lg_d256.npz")
    g, lg, _, _ = synthetic.make_batch(batch_size=1, atoms=10, k=12, seed=5)
    xm, z = GI.features(21, g.num_edges(), 256), GI.features(22, lg.num_edges(), 256)
    assert GI.checksum(xm, z, *lg.edges()) == int(gold["in_crc"])
    out = _conv_run(norm, train, to_oracle(lg), xm, z, 256, 200, torch.float64)
    for k in ("x_out", "y_out", "gx", "gy", "g.edge_gate.weight", "g.src_gate.bias", "g.bn_edges.weight",
              "g.bn_nodes.bias", "g.dst_update.weight"):
        np.testing.assert_allclose(GI.sample(out[k]), gold[f"{tag}.{k}"], rtol=1e-5, atol=1e-6, err_msg=k)


def _small_cases():
    a = synthetic.make_batch(batch_size=3, atoms=9, k=12, seed=31, vary_atoms=True)
    b = synthetic.make_batch(batch_size=2, atoms=6, k=6, seed=32, regular=False)
    return {"reg": a, "knn": b}


SMALL_CFG = dict(alignn_layers=2, gcn_layers=2, hidden_features=64, embedding_features=32)
GRAD_KEYS = ("g.fc.weight", "g.atom_embedding.layer.0.weight", "g.alignn_layers.0.edge_update.edge_gate.weight",
             "g.alignn_layers.1.node_update.src_gate.weight", "g.gcn_layers.1.dst_update.bias",
             "g.alignn_layers.0.node_update.bn_nodes.weight", "g.gcn_layers.0.bn_edges.bias",
             "g.angle_embedding.1.layer.0.weight")


@pytest.mark.parametrize("case", ["reg", "knn"])
@pytest.mark.parametrize("train", [True, False])
def test_full_alignn_matches_reference_fp64(golden_dir, case, train):
    gold = _load(golden_dir, "alignn_small.npz")
    g, lg, lat, tgt = _small_cases()[case]
    assert GI.checksum(*g.edges(), *lg.edges(), g.edata["r"], g.ndata["atom_features"], lg.edata["h"]) == \
        int(gold[f"{case}.in_crc"])
    assert [g.num_nodes(), g.num_edges(), lg.num_edges()] == gold[f"{case}.shape"].tolist()
    dt = torch.float64
    m = O.ALIGNN(norm="batchnorm", **SMALL_CFG).to(dt)
    GI.fill_state_dict(m, 300)
    m.train(train)
    out = m((to_oracle(g, dt), to_oracle(lg, dt), lat.to(dt)))
    loss = (out - tgt.to(dt)).abs().mean()
    grads = dict(zip(["g." + n for n, _ in m.named_parameters()],
                     torch.autograd.grad(loss, list(m.parameters()), allow_unused=True)))
    tag = f"{case}.{'train' if train else 'eval'}"
    np.testing.assert_allclose(out.detach().numpy(), gold[tag + ".out"], rtol=1e-9, atol=1e-10)
    for k in GRAD_KEYS:
        got = grads[k]
        got = np.zeros_like(gold[f"{tag}.{k}"]) if got is None else got.numpy()
        np.testing.assert_allclose(got, gold[f"{tag}.{k}"], rtol=1e-8, atol=1e-10, err_msg=k)


def test_atomwise_energy_forces_match_reference(golden_dir):
    gold = _load(golden_dir, "atomwise_small.npz")
    g, lg, lat, _ = synthetic.make_batch(batch_size=2, atoms=8, k=12, seed=41, vary_atoms=True)
    assert GI.checksum(*g.edges(), *lg.edges(), g.edata["r"], g.ndata["atom_features"]) == int(gold["in_crc"])
    dt = torch.float64
    m = O.ALIGNN(norm="layernorm", **SMALL_CFG).to(dt)
    # same state_dict order as ALIGNNAtomWise for the shared modules
    GI.fill_state_dict(m, 400)
    out, forces, pair = O.energy_and_forces(m, to_oracle(g, dt), to_oracle(lg, dt))
    np.testing.assert_allclose(out.numpy(), gold["out"], rtol=1e-9, atol=1e-10)
    np.testing.assert_allclose(forces.numpy(), gold["forces"], rtol=1e-8, atol=1e-10)
    np.testing.assert_allclose(pair.numpy(), gold["pair_forces"], rtol=1e-8, atol=1e-10)


CUTOFF_CASES = {"mult": dict(use_cutoff_function=True, multiply_cutoff=True, inner_cutoff=2.5, exponent=5),
                "repl": dict(use_cutoff_function=True, multiply_cutoff=False, inner_cutoff=2.5, exponent=3),
                "leak": dict(use_cutoff_function=False, penalty_threshold=1.2)}


@pytest.mark.parametrize("tag", sorted(CUTOFF_CASES))
def test_atomwise_cutoff_and_penalty_variants_match_reference(golden_dir, tag):
    """Cutoff envelope (alignn_atomwise.py:434-451, both `multiply_cutoff` settings) and the short-bond penalty that the
    reference adds in place to `out` when energy_mult_natoms=False (SURVEY App. D-12), on bonds shortened to 0.5-2.8 A."""
    gold = _load(golden_dir, "atomwise_cutoff.npz")
    g, lg, lat, _ = synthetic.make_batch(batch_size=2, atoms=8, k=12, seed=41, vary_atoms=True)
    dt = torch.float64
    m = O.ALIGNN(norm="layernorm", **SMALL_CFG).to(dt)
    GI.fill_state_dict(m, 400)
    og = to_oracle(g, dt)
    og.edata["r"] = og.edata["r"] * 0.35
    out, forces, _ = O.energy_and_forces(m, og, to_oracle(lg, dt), energy_mult_natoms=tag != "leak", **CUTOFF_CASES[tag])
    np.testing.assert_allclose(out.numpy(), gold[tag + ".out"], rtol=1e-9, atol=1e-10)
    np.testing.assert_allclose(forces.numpy(), gold[tag + ".forces"], rtol=1e-8, atol=1e-9)


def test_cutoff_function_of_the_product_matches_oracle():
    from alignn_b200.alignn_atomwise import cutoff_function_based_edges
    r = torch.linspace(0.0, 5.0, 101, dtype=torch.float64)
    for p, rc in ((3, 4.0), (5, 2.5)):
        np.testing.assert_allclose(cutoff_function_based_edges(r, rc, p).numpy(), O.cutoff_envelope(r, rc, p).numpy(), rtol=0, atol=0)


def test_virial_stress_matches_reference(golden_dir):
    """Batched virial stress (alignn_atomwise.py:610-635) from the reference's own pair forces: the oracle loop and
    the product's segment-sum formulation (a device-agnostic torch tail, no kernel of ours) both reproduce it."""
    from alignn_b200.alignn_atomwise import virial_stress
    gold = _load(golden_dir, "atomwise_stress.npz")
    g, lg, lat, _ = synthetic.make_batch(batch_size=2, atoms=8, k=12, seed=41, vary_atoms=True)
    vols = GI.cell_volumes(g.batch_num_nodes())
    assert GI.checksum(*g.edges(), g.edata["r"], vols) == int(gold["in_crc"])
    pair = torch.from_numpy(gold["pair_forces"])
    st = O.virial_stress(to_oracle(g, torch.float64), pair, vols.double(), stress_multiplier=10.0)
    np.testing.assert_allclose(st.numpy(), gold["stresses"], rtol=1e-10, atol=1e-12)
    st2 = virial_stress(g.edata["r"].double(), pair, g.node_graph_offsets(), g.batch_num_edges(), vols, 10.0)
    np.testing.assert_allclose(st2.numpy(), gold["stresses"], rtol=1e-10, atol=1e-12)
    # a symmetric-looking sanity property: crystal b's stress scales as 1 / V_b
    st3 = virial_stress(g.edata["r"].double(), pair, g.node_graph_offsets(), g.batch_num_edges(), 2 * vols, 10.0)
    np.testing.assert_allclose(2 * st3.numpy(), gold["stresses"], rtol=1e-10, atol=1e-12)


# ---- the reference's own property tests for this path, restated (test_force_reduction.py) ----------
class _Simple(torch.nn.Module):
    def __init__(self, width=16):
        super().__init__()
        self.edge_embedding = torch.nn.Linear(1, width)
        self.hidden1 = O.EdgeGatedGraphConv(width, width)
        self.hidden2 = O.EdgeGatedGraphConv(width, width)
        self.fc = torch.nn.Linear(width, 1)
        self.width = width

    def energy(self, pos, s, t):
        bondvec = pos[t] - pos[s]
        y = self.edge_embedding(torch.norm(bondvec, dim=1).unsqueeze(-1))
        x = torch.ones(pos.shape[0], self.width, dtype=pos.dtype)
        g = O.OGraph(s, t, pos.shape[0])
        x, y = self.hidden1(g, x, y)
        x, y = self.hidden2(g, x, y)
        return self.fc(x).sum(), bondvec


def _simple_setup(golden_dir):
    jv = _load(golden_dir, "jvasp_98225.npz")
    pos = torch.from_numpy(jv["coords"])
    m = _Simple().double()
    GI.fill_state_dict(m, 500)
    return m, pos, torch.from_numpy(jv["src"]), torch.from_numpy(jv["dst"])


def test_position_and_displacement_forces_agree(golden_dir):
    """test_force_reduction.py:212-229: dE/dpos == reduction of dE/dbondvec over in- and out-edges."""
    m, pos, s, t = _simple_setup(golden_dir)
    gold = _load(golden_dir, "force_reduction.npz")
    p = pos.clone().requires_grad_(True)
    e, bondvec = m.energy(p, s, t)
    f_x = -torch.autograd.grad(e, p, retain_graph=True)[0]
    pf = -torch.autograd.grad(e, bondvec)[0]
    z = torch.zeros(32, 3, dtype=torch.float64)
    f_vec = z.index_add(0, t, pf) - z.index_add(0, s, pf)
    assert torch.isclose(f_x, f_vec).all()
    np.testing.assert_allclose(e.item(), gold["energy"], rtol=1e-10)
    np.testing.assert_allclose(f_x.numpy(), gold["forces"], rtol=1e-8, atol=1e-10)


def test_forces_match_finite_difference(golden_dir):
    """test_force_reduction.py:233-271 (delta=1e-6, atol 1e-5, rtol 1e-3); a 12-component sample."""
    m, pos, s, t = _simple_setup(golden_dir)
    m.eval()   # fixed statistics so that the energy is a smooth function of one atom's position
    p = pos.clone().requires_grad_(True)
    e, _ = m.energy(p, s, t)
    f_x = -torch.autograd.grad(e, p)[0]
    with torch.no_grad():
        for i in (0, 7, 19, 31):
            for j in range(3):
                pa, pb = pos.clone(), pos.clone()
                pa[i, j] -= 1e-6
                pb[i, j] += 1e-6
                fd = -(m.energy(pb, s, t)[0] - m.energy(pa, s, t)[0]) / 2e-6
                assert torch.isclose(f_x[i, j], fd, atol=1e-5, rtol=1e-3), (i, j, f_x[i, j].item(), fd.item())


def test_conv_two_formulations_agree():
    """index_add formulation (oracle) vs dense-adjacency formulation on a small multigraph."""
    g, _, _, _ = synthetic.make_batch(batch_size=1, atoms=7, k=6, seed=9, regular=False)
    og = to_oracle(g)
    d = 32
    conv = O.EdgeGatedGraphConv(d, d, norm="layernorm").double()
    GI.fill_state_dict(conv, 1)
    x, y = GI.features(1, og.n, d).double(), GI.features(2, og.num_edges(), d).double()
    xo, yo = conv(og, x, y)
    E, N = og.num_edges(), og.n
    inc_dst = torch.zeros(N, E, dtype=torch.float64)
    inc_dst[og.dst, torch.arange(E)] = 1
    inc_src = torch.zeros(E, N, dtype=torch.float64)
    inc_src[torch.arange(E), og.src] = 1
    m = inc_src @ conv.src_gate(x) + inc_dst.t() @ conv.dst_gate(x) + conv.edge_gate(y)
    sig = torch.sigmoid(m)
    h = (inc_dst @ ((inc_src @ conv.dst_update(x)) * sig)) / (inc_dst @ sig + 1e-6)
    x2 = x + torch.nn.functional.silu(conv.bn_nodes(conv.src_update(x) + h))
    y2 = y + torch.nn.functional.silu(conv.bn_edges(m))
    assert torch.allclose(xo, x2, rtol=1e-12, atol=1e-12) and torch.allclose(yo, y2, rtol=1e-12, atol=1e-12)


def test_oracle_only_synthetic_batch_equals_the_product_generator():
    """bench.py's CPU reference arm builds its inputs without importing the product: same graphs, same features."""
    from alignn_b200 import synthetic
    from oracle import synthetic_inputs as SI
    g, lg, lat, tgt = synthetic.make_batch(batch_size=3, atoms=9, k=12, seed=31)
    og, olg, olat, otgt = SI.make_batch(batch_size=3, atoms=9, k=12, seed=31)
    s, d = g.edges()
    assert torch.equal(s.long(), og.src) and torch.equal(d.long(), og.dst)
    assert torch.equal(g.ndata["atom_features"], og.ndata["atom_features"]) and torch.equal(g.edata["r"], og.edata["r"])
    assert torch.equal(lat, olat) and torch.equal(tgt, otgt)
    # L(g): same edge SET (the product emits destination-major, the oracle source-major) with the same cosines
    ls, ld = lg.edges()
    a = sorted(zip(ls.tolist(), ld.tolist(), lg.edata["h"].tolist()))
    b = sorted(zip(olg.src.tolist(), olg.dst.tolist(), olg.edata["h"].tolist()))
    assert a == b
