"""Generate tests/golden/*.npz by running the UNMODIFIED reference model code.

Run in the authoring container only (needs /root/reference, read-only):

    python oracle/make_golden.py

The reference modules alignn/models/alignn.py and alignn/models/alignn_atomwise.py are
imported as they lie under /root/reference.  Their third-party imports that are absent
here are satisfied by stand-ins: `dgl` -> oracle/dgl_stub (DGL's published message
passing semantics in pure torch), `jarvis.*` / `matplotlib` -> empty placeholder modules
(only needed for `import` statements; no jarvis code is on the path under test).

Each fixture stores the reference's OUTPUTS; inputs are re-derived from seeds by
oracle/golden_inputs.py (a crc32 of the inputs is stored to detect drift).  The conv
fixtures store every output as golden_inputs.sample(), at most 4096 elements each, which
keeps every file under 1 MB.  The script
also asserts that the oracle restatement (oracle/alignn_oracle.py) reproduces the
reference to fp64 round-off before anything is written.
"""
import ast
import os
import sys
import types
from unittest import mock

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle", "dgl_stub"))
sys.path.insert(0, REF)

for name in ["jarvis", "jarvis.core", "jarvis.core.atoms", "jarvis.core.specie", "jarvis.core.utils",
             "jarvis.analysis", "jarvis.analysis.structure", "jarvis.analysis.structure.neighbors",
             "matplotlib", "matplotlib.pyplot"]:
    sys.modules.setdefault(name, mock.MagicMock(name=name))

import dgl  # noqa: E402  (the stub)
from alignn.models import alignn as ref_alignn  # noqa: E402
from alignn.models import alignn_atomwise as ref_atomwise  # noqa: E402

from oracle import alignn_oracle as O  # noqa: E402
from oracle import golden_inputs as GI  # noqa: E402
from alignn_b200 import synthetic  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
os.makedirs(OUT, exist_ok=True)


def jvasp_coords():
    src = open(os.path.join(REF, "alignn/tests/test_force_reduction.py")).read()
    tree = ast.parse(src)
    for node in tree.body:
        if isinstance(node, ast.Assign) and getattr(node.targets[0], "id", "") == "jvasp_98225_data":
            data = ast.literal_eval(node.value)
            assert data["cartesian"] is True
            return np.asarray(data["coords"], dtype=np.float64)
    raise RuntimeError("fixture not found")


def to_dgl(g):
    """alignn_b200.Graph -> stub DGLGraph (same node/edge order)."""
    s, d = g.edges()
    dg = dgl.DGLGraph(s.long(), d.long(), g.num_nodes(), g.batch_num_nodes().clone(), g.batch_num_edges().clone())
    dg.ndata.update(g.ndata)
    dg.edata.update(g.edata)
    return dg


def to_oracle(g):
    s, d = g.edges()
    og = O.OGraph(s.long(), d.long(), g.num_nodes(), g.batch_num_nodes(), g.batch_num_edges())
    og.ndata.update(g.ndata)
    og.edata.update(g.edata)
    return og


def npd(d):
    return {k: (v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)) for k, v in d.items()}


def conv_case(ref_cls, norm, train, g_dgl, g_or, x, y, d, seed, dtype):
    """Run one reference EdgeGatedGraphConv + the oracle twin; return outputs and grads."""
    ref = ref_cls(d, d).to(dtype)
    GI.fill_state_dict(ref, seed)
    orc = O.EdgeGatedGraphConv(d, d, norm=norm).to(dtype)
    orc.load_state_dict(ref.state_dict())
    ref.train(train)
    orc.train(train)
    wx = GI.features(seed + 1, x.shape[0], d).to(dtype)
    wy = GI.features(seed + 2, y.shape[0], d).to(dtype)
    res = []
    for mod, gg in ((ref, g_dgl), (orc, g_or)):
        xi = x.to(dtype).clone().requires_grad_(True)
        yi = y.to(dtype).clone().requires_grad_(True)
        xo, yo = mod(gg, xi, yi)
        loss = (xo * wx).sum() + (yo * wy).sum()
        grads = torch.autograd.grad(loss, [xi, yi] + list(mod.parameters()))
        out = {"x_out": xo, "y_out": yo, "gx": grads[0], "gy": grads[1]}
        for (n, _), gr in zip(mod.named_parameters(), grads[2:]):
            out["g." + n] = gr
        if norm == "batchnorm":
            out["bn_nodes.running_mean"] = mod.bn_nodes.running_mean.clone()
            out["bn_nodes.running_var"] = mod.bn_nodes.running_var.clone()
            out["bn_edges.running_mean"] = mod.bn_edges.running_mean.clone()
            out["bn_edges.running_var"] = mod.bn_edges.running_var.clone()
        res.append(out)
    return res


def check_close(a, b, tol, what):
    for k in a:
        err = (a[k] - b[k]).abs().max().item()
        ref = b[k].abs().max().item() + 1e-30
        assert err <= tol * max(ref, 1.0), f"{what}:{k}: oracle deviates from reference by {err} (scale {ref})"


def main():
    torch.manual_seed(0)
    # ---------------------------------------------------------------- jvasp conv (config 1 shape)
    coords = jvasp_coords()
    pos = torch.from_numpy(coords)
    dg = dgl.radius_graph(pos, 5.0)
    s, dd = dg.edges()
    np.savez(os.path.join(OUT, "jvasp_98225.npz"), coords=coords, src=s.numpy(), dst=dd.numpy())
    og = O.OGraph(s, dd, 32)
    E = s.numel()
    d = 64
    x = GI.features(11, 32, d)
    y = GI.features(12, E, d)
    store = {"in_crc": GI.checksum(x, y, s, dd)}
    for tag, ref_cls, norm, train in (("bn_train", ref_alignn.EdgeGatedGraphConv, "batchnorm", True),
                                      ("bn_eval", ref_alignn.EdgeGatedGraphConv, "batchnorm", False),
                                      ("ln", ref_atomwise.EdgeGatedGraphConv, "layernorm", True)):
        r64, o64 = conv_case(ref_cls, norm, train, dg, og, x, y, d, 100, torch.float64)
        check_close(o64, r64, 1e-12, f"jvasp {tag} fp64")
        r32, o32 = conv_case(ref_cls, norm, train, dg, og, x, y, d, 100, torch.float32)
        check_close(o32, r32, 2e-5, f"jvasp {tag} fp32")
        for k, v in npd(r64).items():
            store[f"{tag}.{k}"] = GI.sample(v)
    np.savez_compressed(os.path.join(OUT, "conv_jvasp_d64.npz"), **store)
    print("conv_jvasp_d64: E =", E)

    # ---------------------------------------------------------------- d=256 conv on a line graph
    g, lg, lat, tgt = synthetic.make_batch(batch_size=1, atoms=10, k=12, seed=5)
    d = 256
    xm = GI.features(21, g.num_edges(), d)          # L(g) node features (= bond features m)
    z = GI.features(22, lg.num_edges(), d)
    ldg, log_ = to_dgl(lg), to_oracle(lg)
    store = {"in_crc": GI.checksum(xm, z, *lg.edges())}
    for tag, ref_cls, norm, train in (("bn_train", ref_alignn.EdgeGatedGraphConv, "batchnorm", True),
                                      ("bn_eval", ref_alignn.EdgeGatedGraphConv, "batchnorm", False),
                                      ("ln", ref_atomwise.EdgeGatedGraphConv, "layernorm", True)):
        r64, o64 = conv_case(ref_cls, norm, train, ldg, log_, xm, z, d, 200, torch.float64)
        check_close(o64, r64, 1e-12, f"lg256 {tag} fp64")
        for k in ("x_out", "y_out", "gx", "gy", "g.edge_gate.weight", "g.src_gate.bias", "g.bn_edges.weight",
                  "g.bn_nodes.bias", "g.dst_update.weight"):
            store[f"{tag}.{k}"] = GI.sample(r64[k])
    np.savez_compressed(os.path.join(OUT, "conv_lg_d256.npz"), **store)
    print("conv_lg_d256: E =", g.num_edges(), "T =", lg.num_edges())

    # ---------------------------------------------------------------- full ALIGNN (BatchNorm), small
    g, lg, lat, tgt = synthetic.make_batch(batch_size=3, atoms=9, k=12, seed=31, vary_atoms=True)
    g2, lg2, lat2, tgt2 = synthetic.make_batch(batch_size=2, atoms=6, k=6, seed=32, regular=False)
    cases = {"reg": (g, lg, lat, tgt), "knn": (g2, lg2, lat2, tgt2)}
    cfg = dict(alignn_layers=2, gcn_layers=2, hidden_features=64, embedding_features=32)
    store = {}
    for cname, (g, lg, lat, tgt) in cases.items():
        store[f"{cname}.in_crc"] = GI.checksum(*g.edges(), *lg.edges(), g.edata["r"], g.ndata["atom_features"], lg.edata["h"])
        store[f"{cname}.shape"] = np.asarray([g.num_nodes(), g.num_edges(), lg.num_edges()])
        for dtype, dn in ((torch.float64, "f64"),):
            ref = ref_alignn.ALIGNN(ref_alignn.ALIGNNConfig(name="alignn", **cfg)).to(dtype)
            GI.fill_state_dict(ref, 300)
            orc = O.ALIGNN(norm="batchnorm", **cfg).to(dtype)
            orc.load_state_dict(ref.state_dict())
            for train in (True, False):
                GI.fill_state_dict(ref, 300)          # fresh running statistics for each mode
                orc.load_state_dict(ref.state_dict())
                outs = []
                for mod, conv in ((ref, to_dgl), (orc, to_oracle)):
                    mod.train(train)
                    gg, ll = conv(g), conv(lg)
                    for t in (gg, ll):
                        for dct in (t.ndata, t.edata):
                            for k in list(dct):
                                if dct[k].is_floating_point():
                                    dct[k] = dct[k].to(dtype)
                    out = mod((gg, ll, lat.to(dtype)))
                    loss = (out - tgt.to(dtype)).abs().mean()          # L1, train.py:240
                    grads = torch.autograd.grad(loss, [p for p in mod.parameters()], allow_unused=True)
                    o = {"out": out, "loss": loss}
                    for (n, p), gr in zip(mod.named_parameters(), grads):
                        o["g." + n] = torch.zeros_like(p) if gr is None else gr
                    outs.append(o)
                check_close(outs[1], outs[0], 1e-11, f"alignn {cname} train={train}")
                tag = f"{cname}.{'train' if train else 'eval'}"
                store[tag + ".out"] = outs[0]["out"].detach().numpy()
                store[tag + ".loss"] = outs[0]["loss"].detach().numpy()
                for k in ("g.fc.weight", "g.atom_embedding.layer.0.weight", "g.alignn_layers.0.edge_update.edge_gate.weight",
                          "g.alignn_layers.1.node_update.src_gate.weight", "g.gcn_layers.1.dst_update.bias",
                          "g.alignn_layers.0.node_update.bn_nodes.weight", "g.gcn_layers.0.bn_edges.bias",
                          "g.angle_embedding.1.layer.0.weight"):
                    store[tag + "." + k] = outs[0][k].detach().numpy()
    np.savez_compressed(os.path.join(OUT, "alignn_small.npz"), **store)
    print("alignn_small ok")

    # ---------------------------------------------------------------- ALIGNNAtomWise (LayerNorm): energy + forces
    g, lg, lat, tgt = synthetic.make_batch(batch_size=2, atoms=8, k=12, seed=41, vary_atoms=True)
    acfg = dict(alignn_layers=2, gcn_layers=2, hidden_features=64, embedding_features=32, atom_input_features=92,
                calculate_gradient=True, use_penalty=True, stresswise_weight=0.0)
    dtype = torch.float64
    ref = ref_atomwise.ALIGNNAtomWise(ref_atomwise.ALIGNNAtomWiseConfig(name="alignn_atomwise", **acfg)).to(dtype)
    GI.fill_state_dict(ref, 400)
    orc = O.ALIGNN(norm="layernorm", alignn_layers=2, gcn_layers=2, hidden_features=64, embedding_features=32).to(dtype)
    missing = orc.load_state_dict(ref.state_dict(), strict=False)
    assert not missing.missing_keys, missing
    gg, ll = to_dgl(g), to_dgl(lg)
    for t in (gg, ll):
        for dct in (t.ndata, t.edata):
            for k in list(dct):
                if dct[k].is_floating_point():
                    dct[k] = dct[k].to(dtype)
    res = ref((gg, ll, lat.to(dtype)))
    og_, ol_ = to_oracle(g), to_oracle(lg)
    for t in (og_, ol_):
        for dct in (t.ndata, t.edata):
            for k in list(dct):
                if dct[k].is_floating_point():
                    dct[k] = dct[k].to(dtype)
    en, forces, pair = O.energy_and_forces(orc, og_, ol_, energy_mult_natoms=True)
    assert (en - res["out"].detach()).abs().max() < 1e-11
    assert (forces - res["grad"].detach()).abs().max() < 1e-11
    np.savez_compressed(os.path.join(OUT, "atomwise_small.npz"),
                        in_crc=GI.checksum(*g.edges(), *lg.edges(), g.edata["r"], g.ndata["atom_features"]),
                        out=res["out"].detach().numpy(), forces=res["grad"].detach().numpy(),
                        pair_forces=pair.numpy())
    print("atomwise_small ok: E =", g.num_edges(), "T =", lg.num_edges())

    # same batch with the stress head on (alignn_atomwise.py:567-638, batch_stress=True); V = cell volume on every atom
    vols = GI.cell_volumes(g.batch_num_nodes())
    gg.ndata["V"] = vols.to(dtype)
    ref_s = ref_atomwise.ALIGNNAtomWise(ref_atomwise.ALIGNNAtomWiseConfig(
        name="alignn_atomwise", **{**acfg, "stresswise_weight": 0.1, "stress_multiplier": 10.0})).to(dtype)
    GI.fill_state_dict(ref_s, 400)
    res_s = ref_s((gg, ll, lat.to(dtype)))
    assert (res_s["grad"] - res["grad"]).abs().max() < 1e-12
    st = O.virial_stress(og_, pair, vols.to(dtype), stress_multiplier=10.0)
    assert (st - res_s["stresses"].detach()).abs().max() < 1e-11 * st.abs().max()
    np.savez_compressed(os.path.join(OUT, "atomwise_stress.npz"),
                        in_crc=GI.checksum(*g.edges(), g.edata["r"], vols),
                        stresses=res_s["stresses"].detach().numpy(), pair_forces=pair.numpy())
    print("atomwise_stress ok:", tuple(res_s["stresses"].shape))

    # cutoff-envelope variants (alignn_atomwise.py:434-451) and the penalty that leaks into `out` when
    # energy_mult_natoms=False (SURVEY App. D-12); shorter bonds so that envelope and penalty are exercised
    store = {}
    gg.edata["r"] = gg.edata["r"] * 0.35
    og_.edata["r"] = og_.edata["r"] * 0.35
    for tag, extra in (("mult", dict(use_cutoff_function=True, multiply_cutoff=True, inner_cutoff=2.5, exponent=5)),
                       ("repl", dict(use_cutoff_function=True, multiply_cutoff=False, inner_cutoff=2.5, exponent=3)),
                       ("leak", dict(use_cutoff_function=False, penalty_threshold=1.2))):
        cfg_c = {**acfg, "energy_mult_natoms": tag != "leak", **extra}
        ref_c = ref_atomwise.ALIGNNAtomWise(ref_atomwise.ALIGNNAtomWiseConfig(name="alignn_atomwise", **cfg_c)).to(dtype)
        GI.fill_state_dict(ref_c, 400)
        res_c = ref_c((gg, ll, lat.to(dtype)))
        okw = {k: v for k, v in extra.items()}
        en_c, f_c, pair_c = O.energy_and_forces(orc, og_, ol_, energy_mult_natoms=tag != "leak", **okw)
        assert (en_c - res_c["out"].detach()).abs().max() < 1e-10 * max(1.0, float(en_c.abs().max())), tag
        assert (f_c - res_c["grad"].detach()).abs().max() < 1e-10 * max(1.0, float(f_c.abs().max())), tag
        store[tag + ".out"] = res_c["out"].detach().numpy()
        store[tag + ".forces"] = res_c["grad"].detach().numpy()
    np.savez_compressed(os.path.join(OUT, "atomwise_cutoff.npz"),
                        in_crc=GI.checksum(*g.edges(), *lg.edges(), g.edata["r"], g.ndata["atom_features"]), **store)
    print("atomwise_cutoff ok:", {k: float(np.abs(v).max()) for k, v in store.items()})

    # ---------------------------------------------------------------- reference test properties (fp64)
    # tests/test_force_reduction.py:212-229 restated on the real reference conv + stub graph ops.
    torch.set_default_dtype(torch.float64)

    class Simple(torch.nn.Module):
        def __init__(self, conv_cls, width=16):
            super().__init__()
            self.edge_embedding = torch.nn.Linear(1, width)
            self.hidden1 = conv_cls(width, width)
            self.hidden2 = conv_cls(width, width)
            self.fc = torch.nn.Linear(width, 1)
            self.width = width

    m = Simple(ref_alignn.EdgeGatedGraphConv)
    GI.fill_state_dict(m, 500)
    p = pos.clone().requires_grad_(True)
    gph = dgl.radius_graph(p, 5.0)
    s, t_ = gph.edges()
    bondvec = p[t_] - p[s]
    yy = m.edge_embedding(torch.norm(bondvec, dim=1).unsqueeze(-1))
    xx = torch.ones(32, 16)
    xx, yy = m.hidden1(gph, xx, yy)
    xx, yy = m.hidden2(gph, xx, yy)
    e = m.fc(xx).sum()
    f_x = -torch.autograd.grad(e, p, retain_graph=True)[0]
    pf = -torch.autograd.grad(e, bondvec)[0]
    z3 = torch.zeros(32, 3)
    f_vec = z3.index_add(0, t_, pf) - z3.index_add(0, s, pf)
    assert torch.isclose(f_x, f_vec).all()
    np.savez(os.path.join(OUT, "force_reduction.npz"), energy=e.detach().numpy(), forces=f_x.detach().numpy())
    torch.set_default_dtype(torch.float32)
    print("force_reduction property holds on reference conv; golden written")


if __name__ == "__main__":
    main()
