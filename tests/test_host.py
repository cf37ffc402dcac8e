"""CPU tests of the host side: the C-ABI library loads and exports every symbol the header
declares, the ctypes struct mirrors the C struct, the weight export (role permutations) is
right, the synthetic generator is deterministic.  No compute calls (no GPU here)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from helpers import load_fixture, load_golden_weights

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "nabla_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(nb200_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from nabladft_b200 import _lib, build

    build.build()
    lib = _lib.load()
    declared = _declared_symbols()
    assert len(declared) >= 10
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/nabla_b200.h but not exported"
        assert name in _lib.SIGNATURES, f"{name} has no ctypes signature"
    assert lib.nb200_version() == 100


def test_weights_struct_layout_matches_header():
    from nabladft_b200._lib import PainnWeights

    src = open(os.path.join(ROOT, "include", "nabla_b200.h")).read()
    body = src[src.index("typedef struct nb200_painn_weights {"):src.index("} nb200_painn_weights;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for decl in body.split("{", 1)[1].split(";"):
        decl = decl.strip()
        if not decl:
            continue
        decl = re.sub(r"^(const\s+)?(int32_t|float)\s*\*?", "", decl)
        names += [n.strip().lstrip("*").strip() for n in decl.split(",")]
    assert names == [f[0] for f in PainnWeights._fields_]
    assert ctypes.sizeof(PainnWeights) == 4 * 10 + 8 + 4 + 4 + 8 * 16  # no hidden padding surprises


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    from nabladft_b200 import _lib

    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(_lib.NablaB200Error):
        _lib.load()


def test_cpu_input_is_rejected_not_emulated():
    from nabladft_b200._lib import NablaB200Error
    from nabladft_b200.painn_oc import PaiNN

    net = PaiNN(hidden_channels=128, num_layers=2, num_rbf=100, cutoff=5.0, max_neighbors=100, direct_forces=False, use_pbc=False, num_elements=100).eval()

    class D:
        pass

    d = D()
    d.z, d.pos, d.batch = load_fixture([0], torch.float32)
    with pytest.raises(NablaB200Error):
        net(d)


def test_painn_oc_export_matches_oracle():
    from canonical_ref import canonical_energy_forces
    from nabladft_b200.painn_oc import PaiNN
    from oracle.painn_oc import PaiNNOC

    kw = dict(hidden_channels=128, num_layers=3, num_rbf=100, cutoff=5.0, max_neighbors=100, num_elements=100)
    ours = load_golden_weights(PaiNN(direct_forces=False, use_pbc=False, **kw), torch.float32)
    ref = PaiNNOC(**kw).double()
    ref.load_state_dict({k: v.double() for k, v in ours.state_dict().items()}, strict=True)
    z, pos, batch = load_fixture([0, 4])
    e0, f0 = ref(z, pos.clone(), batch)
    t, s = ours._export()
    e1, f1 = canonical_energy_forces(t, s, z, pos, batch)
    assert torch.allclose(e0, e1, atol=1e-5) and torch.allclose(f0, f1, atol=1e-5)  # weights were rounded to fp32


def test_spk_export_matches_oracle_and_state_dict_names():
    from canonical_ref import canonical_energy_forces
    from nabladft_b200 import spk
    from oracle.graph import ase_neighbor_list, batch_to_ptr
    from oracle.spk import NeuralNetworkPotential as OracleNNP
    from oracle.spk import SpkPaiNN

    ours = spk.NeuralNetworkPotential(
        representation=spk.PaiNN(n_atom_basis=128, n_interactions=2, radial_basis=spk.GaussianRBF(n_rbf=100, cutoff=5.0),
                                 cutoff_fn=spk.CosineCutoff(cutoff=5.0)),
        input_modules=[spk.PairwiseDistances()],
        output_modules=[spk.Atomwise(n_in=128, output_key="energy"), spk.Forces()],
        postprocessors=[spk.AddOffsets(property="energy", add_mean=True)],
    )
    load_golden_weights(ours, torch.float32)
    ours.postprocessors[0].mean.fill_(-0.3)
    ref = OracleNNP(SpkPaiNN(n_interactions=2)).double()
    ours_sd = ours.state_dict()
    ref_sd = ref.state_dict()
    # every oracle (== schnetpack 2.0.4) key exists under the same name and shape
    for k, v in ref_sd.items():
        assert k in ours_sd and tuple(ours_sd[k].shape) == tuple(v.shape), k
    ref.load_state_dict({k: ours_sd[k].double() for k in ref_sd}, strict=True)
    z, pos, batch = load_fixture([1, 2])
    idx_i, idx_j = ase_neighbor_list(pos, batch_to_ptr(batch), 5.0)
    out = ref({"_atomic_numbers": z, "_positions": pos.clone(), "_idx_i": idx_i, "_idx_j": idx_j, "_idx_m": batch})
    t, s = ours._export(True)
    e1, f1 = canonical_energy_forces(t, s, z, pos, batch)
    assert torch.allclose(out["energy"], e1, atol=1e-5) and torch.allclose(out["forces"], f1, atol=1e-5)


def test_spk_strict_load_of_schnetpack_shaped_checkpoint():
    """A schnetpack 2.0.4 checkpoint carries `postprocessors.0.atomref` (AddOffsets registers zeros[zmax] even without atomrefs) and the
    cutoff as a buffer; `load_state_dict(strict=True)` must accept it, a non-zero atomref must be refused, and the exported cutoff follows
    the loaded buffer (ADVICE r1)."""
    from nabladft_b200 import spk

    def make():
        return spk.NeuralNetworkPotential(
            representation=spk.PaiNN(n_atom_basis=128, n_interactions=1, radial_basis=spk.GaussianRBF(n_rbf=100, cutoff=5.0),
                                     cutoff_fn=spk.CosineCutoff(cutoff=5.0)),
            input_modules=[spk.PairwiseDistances()], output_modules=[spk.Atomwise(n_in=128, output_key="energy"), spk.Forces()],
            postprocessors=[spk.AddOffsets(property="energy", add_mean=True)])

    sd = make().state_dict()
    assert "postprocessors.0.atomref" in sd and "postprocessors.0.mean" in sd
    sd["postprocessors.0.atomref"] = torch.zeros(87)          # zmax of the training set, not our default length
    sd["representation.cutoff_fn.cutoff"] = torch.tensor([4.5])
    net = make()
    net.load_state_dict(sd, strict=True)
    assert net.postprocessors[0].atomref.shape == (87,)
    _, scalars = net._export(True)
    assert abs(scalars["cutoff"] - 4.5) < 1e-7
    sd["postprocessors.0.atomref"] = torch.ones(87)
    with pytest.raises(NotImplementedError):
        make().load_state_dict(sd, strict=True)


def test_synth_is_seeded_and_druglike():
    from nabladft_b200.synth import synth_batch

    a, b = synth_batch(3, 8), synth_batch(3, 8)
    assert all(np.array_equal(a[k], b[k]) for k in a)
    n = np.diff(a["mol_ptr"])
    heavy = [int((a["z"][a["mol_ptr"][m]:a["mol_ptr"][m + 1]] > 1).sum()) for m in range(8)]
    assert max(heavy) <= 30 and min(heavy) >= 5 and n.max() <= 64
    for m in range(8):
        p = a["pos"][a["mol_ptr"][m]:a["mol_ptr"][m + 1]].astype(np.float64)
        d = np.linalg.norm(p[:, None] - p[None], axis=-1) + np.eye(len(p)) * 10
        assert d.min() > 0.9


def test_b200_model_yamls_instantiate():
    """config/model/*-b200.yaml: the Hydra `_target_` seam resolves to our classes (minimal resolver; hydra is absent)."""
    import importlib

    import yaml

    def inst(node):
        if isinstance(node, dict):
            kw = {k: inst(v) for k, v in node.items() if k != "_target_"}
            if "_target_" in node:
                mod, name = node["_target_"].rsplit(".", 1)
                return getattr(importlib.import_module(mod), name)(**kw)
            return kw
        if isinstance(node, list):
            return [inst(v) for v in node]
        return node

    for fn, cls in (("painn-oc-b200.yaml", "PaiNN"), ("painn-b200.yaml", "NeuralNetworkPotential"), ("schnet-b200.yaml", "NeuralNetworkPotential")):
        cfg = yaml.safe_load(open(os.path.join(ROOT, "config", "model", fn)))
        model = inst(cfg["model"])
        assert type(model).__name__ == cls and sum(p.numel() for p in model.parameters()) > 100000

    # the files are COMPLETE copies of the reference's model yamls (pipelines.py:104 instantiates the whole node: task, optimizer,
    # scheduler, losses, metric, ema), with only the model-class targets swapped -- top-level keys as in config/model/<name>.yaml
    spk_keys = ["_target_", "model_name", "model", "outputs", "optimizer_cls", "optimizer_args", "scheduler_cls", "scheduler_args", "scheduler_monitor"]
    pyg_keys = ["_target_", "model_name", "net", "optimizer", "lr_scheduler", "losses", "loss_coefs", "metric"]
    top = {"painn-b200.yaml": spk_keys, "schnet-b200.yaml": spk_keys, "painn-oc-b200.yaml": [k if k != "net" else "model" for k in pyg_keys],
           "qhnet-b200.yaml": pyg_keys + ["ema"], "gemnet-oc-b200.yaml": pyg_keys}
    # key-for-key against the reference files as parsed (tests/golden/make_reference_samples.py)
    refs = yaml.safe_load(open(os.path.join(ROOT, "tests", "golden", "reference_model_configs.yaml")))
    assert len(refs) == len(top)
    for fn, keys in top.items():
        cfg = yaml.safe_load(open(os.path.join(ROOT, "config", "model", fn)))
        assert list(cfg.keys()) == keys, fn
        ref = refs[fn.replace("-b200", "")]
        assert list(cfg.keys()) == list(ref.keys()), fn

        def strip(node):  # compare everything except the swapped model-class targets
            if isinstance(node, dict):
                return {k: ("<cls>" if k == "_target_" and str(v).startswith(("nabladft_b200.", "schnetpack.", "nablaDFT.")) else strip(v))
                        for k, v in node.items()}
            return [strip(v) for v in node] if isinstance(node, list) else node

        assert strip(cfg) == strip(ref), fn


def test_schnet_export_matches_oracle_and_state_dict_names():
    from nabladft_b200 import spk
    from oracle.graph import ase_neighbor_list, batch_to_ptr
    from oracle.spk import NeuralNetworkPotential as OracleNNP
    from oracle.spk import SpkSchNet

    ours = spk.NeuralNetworkPotential(
        representation=spk.SchNet(n_atom_basis=128, n_interactions=3, radial_basis=spk.GaussianRBF(n_rbf=100, cutoff=5.0),
                                  cutoff_fn=spk.CosineCutoff(cutoff=5.0)),
        input_modules=[spk.PairwiseDistances()], output_modules=[spk.Atomwise(n_in=128, output_key="energy"), spk.Forces()],
        postprocessors=[spk.AddOffsets(property="energy", add_mean=True)])
    load_golden_weights(ours, torch.float32)
    ref = OracleNNP(SpkSchNet(n_interactions=3)).double()
    ours_sd, ref_sd = ours.state_dict(), ref.state_dict()
    for k, v in ref_sd.items():
        assert k in ours_sd and tuple(ours_sd[k].shape) == tuple(v.shape), k
    ref.load_state_dict({k: ours_sd[k].double() for k in ref_sd}, strict=True)
    t, s = ours._export(True)
    # canonical evaluation of the SchNet export on CPU (mirrors schnet.cu)
    z, pos, batch = load_fixture([1, 2])
    idx_i, idx_j = ase_neighbor_list(pos, batch_to_ptr(batch), 5.0)
    out = ref({"_atomic_numbers": z, "_positions": pos.clone(), "_idx_i": idx_i, "_idx_j": idx_j, "_idx_m": batch})
    import math
    P = pos.clone().requires_grad_(True)
    td = {k: v.double() for k, v in t.items()}
    r = P[idx_j] - P[idx_i]
    d = r.norm(dim=1)
    phi = torch.exp(s["rbf_coeff"] * (d[:, None] - td["rbf_offsets"][None]) ** 2)
    fc = 0.5 * (torch.cos(d * math.pi / s["cutoff"]) + 1)
    ssp = lambda x: torch.nn.functional.softplus(x) - math.log(2.0)
    x = td["emb"][z]
    for l in range(s["n_layers"]):
        W = (ssp(phi @ td["w_f1"][l] + td["b_f1"][l]) @ td["W_f2"][l].T + td["b_f2"][l]) * fc[:, None]
        y = x @ td["I1"][l].T
        agg = torch.zeros_like(x).index_add_(0, idx_i, y[idx_j] * W)
        x = x + ssp(agg @ td["P1"][l].T + td["p1"][l]) @ td["P2"][l].T + td["p2"][l]
    eps = torch.nn.functional.silu(x @ td["R1"].T + td["e1"]) @ td["R2"].T + td["e2"]
    e = torch.zeros(2, dtype=torch.float64).index_add_(0, batch, eps.squeeze(-1))
    f = -torch.autograd.grad(e.sum(), P)[0]
    e = e + s["energy_shift_per_atom"] * torch.bincount(batch).double()
    assert torch.allclose(out["energy"], e.detach(), atol=1e-5) and torch.allclose(out["forces"], f, atol=1e-5)


def test_losses_match_reference_formulas():
    """HamiltonianLoss on packed per-molecule matrices == the reference formula on the dense block diagonal
    (nablaDFT/qhnet/loss.py:9-16 with masks = block_diag(ones), qhnet.py:368-373); L2Loss (gemnet_oc/loss.py:5-22)."""
    from nabladft_b200.losses import HamiltonianLoss, L2Loss

    g = torch.Generator().manual_seed(0)
    preds = [torch.randn(n, n, generator=g, dtype=torch.float64) for n in (7, 12, 5)]
    targs = [torch.randn(n, n, generator=g, dtype=torch.float64) for n in (7, 12, 5)]
    P, T = torch.block_diag(*preds), torch.block_diag(*targs)
    M = torch.block_diag(*[torch.ones_like(t) for t in targs])
    diff = P - T
    ref = torch.sqrt(torch.mean(diff**2) * P.numel() / M.sum()) + torch.mean(diff.abs()) * P.numel() / M.sum()
    loss = HamiltonianLoss()
    assert torch.allclose(loss(preds, targs), ref) and torch.allclose(loss(P, T, M), ref)
    f, t = torch.randn(9, 3, generator=g), torch.randn(9, 3, generator=g)
    assert torch.allclose(L2Loss()(f, t), (f - t).norm(dim=-1).mean())
    # the Hamiltonian metric of a step: MaskedMeanAbsoluteError (masked_mae.py:12-20: sum|dH| / count_nonzero(target) over the dense
    # block diagonal) times norm_coef = numel / mask.sum (qhnet.py:490-495); a target with exact zeros inside a block exercises the mask
    from nabladft_b200.losses import masked_mae

    targs[1][2, 3] = 0.0
    T = torch.block_diag(*targs)
    ref_metric = (P - T).abs().sum() / torch.count_nonzero(T) * (P.numel() / M.sum())
    assert torch.allclose(masked_mae(preds, targs), ref_metric)
    assert torch.allclose(masked_mae(preds[:1], targs[:1]), (preds[0] - targs[0]).abs().sum() / torch.count_nonzero(targs[0]))


def test_optimization_host_logic():
    import numpy as np
    import pytest
    import yaml

    from nabladft_b200 import optimization as opt
    from nabladft_b200._lib import NablaB200Error

    assert abs(opt.convert_units("eV", "Hartree") - 1 / 27.211386245988) < 1e-15
    assert opt.convert_units("Hartree", "Hartree") == 1.0 and opt.convert_units("Ang", "Angstrom") == 1.0
    assert abs(opt.convert_units("Bohr", "Angstrom") - 0.529177210903) < 1e-15
    with pytest.raises(ValueError):
        opt.convert_units("eV", "Angstrom")
    a = opt.SimpleAtoms(np.zeros((3, 3)), [1, 6, 8])
    b = a.copy()
    assert a == b and len(a) == 3
    b.positions[0, 0] = 1.0
    assert a != b
    moved = opt._like(a, np.ones((3, 3)))
    assert isinstance(moved, opt.SimpleAtoms) and np.array_equal(moved.get_atomic_numbers(), [1, 6, 8]) and moved.get_positions()[2, 2] == 1.0
    with pytest.raises(NablaB200Error):  # no CPU fallback
        opt.PyGBatchwiseCalculator(torch.nn.Identity(), device="cpu")
    here = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for rel, cls in (("config/optimizer/batchwise_lbfgs-b200.yaml", "ASEBatchwiseLBFGS"), ("config/calculator/pyg_calculator-b200.yaml", "PyGBatchwiseCalculator"),
                     ("config/calculator/spk_calculator-b200.yaml", "SpkBatchwiseCalculator")):
        cfg = yaml.safe_load(open(os.path.join(here, rel)))
        mod, name = cfg["_target_"].rsplit(".", 1)
        assert mod == "nabladft_b200.optimization" and name == cls and hasattr(opt, name)


def test_training_autograd_bridge_routes_canonical_gradients_to_named_parameters():
    """CPU check of nabladft_b200/training.py with a stand-in engine: whatever gradient the engine reports for the CANONICAL tensors must
    arrive on the reference-named parameters exactly as autograd would carry it through the export permutations (chunk swaps of
    PaiNN-OC, the [L*3n, K] -> [L, K, 3n] view of the schnetpack filter net)."""
    from nabladft_b200 import spk
    from nabladft_b200.painn_oc import PaiNN
    from nabladft_b200.training import energy_forces_training

    class FakeEngine:
        """follows engine.PainnEngine's two-call training step: the forward keeps a token, the backward call uses the kept state while the
        token is current and the weights key is the forward's; `drop_kept` simulates another launch in between (one-call fallback)."""

        def __init__(self, drop_kept=False):
            self._wkey, self.calls, self.kinds, self._token, self.drop_kept = None, [], [], 0, drop_kept

        def set_weights(self, key, tensors, scalars):
            self.tensors, self._wkey = tensors, key

        def run_train_forward(self, z, pos, mol_ptr, n_mol):  # the forward of the training bridge (status check deferred)
            self._token += 1
            return torch.arange(n_mol, dtype=torch.float32), torch.zeros(z.shape[0], 3), self._token

        def kept(self, token):
            return token == self._token and not self.drop_kept

        def _grads(self, seed, force_seed):
            self.calls.append((seed.clone(), None if force_seed is None else force_seed.clone()))
            g = torch.Generator().manual_seed(11)
            return {k: torch.randn(v.shape, generator=g) * float(seed.sum()) for k, v in self.tensors.items() if k != "rbf_offsets"}

        def run_train_backward(self, token, z, mol_ptr, seed, force_seed):
            assert self.kept(token)
            self.kinds.append("kept")
            return self._grads(seed, force_seed)

        def run_train(self, z, pos, mol_ptr, n_mol, seed, force_seed):
            self.kinds.append("recompute")
            return None, None, self._grads(seed, force_seed)

    z, pos, mol_ptr = torch.tensor([1, 6, 8], dtype=torch.int32), torch.zeros(3, 3), torch.tensor([0, 2, 3], dtype=torch.int32)
    oc = PaiNN(hidden_channels=128, num_layers=2, num_rbf=100, cutoff=5.0, max_neighbors=100, direct_forces=False, use_pbc=False, num_elements=100)
    nnp = spk.NeuralNetworkPotential(
        representation=spk.PaiNN(n_atom_basis=128, n_interactions=2, radial_basis=spk.GaussianRBF(n_rbf=100, cutoff=5.0), cutoff_fn=spk.CosineCutoff(cutoff=5.0)),
        input_modules=[spk.PairwiseDistances()], output_modules=[spk.Atomwise(n_in=128, output_key="energy"), spk.Forces()])
    for model, export, drop in ((oc, lambda m: m._export_impl(detach=False), False), (nnp, lambda m: m._export_impl(False, detach=False), True)):
        eng = FakeEngine(drop_kept=drop)
        tensors, scalars = export(model)
        e, f = energy_forces_training(eng, tensors, scalars, z, pos, mol_ptr, 2)
        seed = torch.tensor([0.5, -2.0])
        (seed * e).sum().backward()
        got = {k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None}
        assert torch.equal(eng.calls[0][0], seed) and eng.calls[0][1] is None
        # expected: the same canonical gradients pushed through the export graph by autograd alone
        model.zero_grad()
        tensors2, _ = export(model)
        g = torch.Generator().manual_seed(11)
        canon = {k: torch.randn(v.shape, generator=g) * float(seed.sum()) for k, v in tensors.items() if k != "rbf_offsets"}
        torch.autograd.backward([tensors2[k] for k in canon], [canon[k] for k in canon])
        want = {k: p.grad for k, p in model.named_parameters() if p.grad is not None}
        assert set(got) == set(want) and len(got) >= 16
        assert all(torch.equal(got[k], want[k]) for k in want)
        # the force seed is handed to the engine untouched
        model.zero_grad()
        tensors3, _ = export(model)
        e, f = energy_forces_training(eng, tensors3, scalars, z, pos, mol_ptr, 2)
        w = torch.arange(9, dtype=torch.float32).view(3, 3)
        (f * w).sum().backward()
        assert torch.equal(eng.calls[-1][1], w) and float(eng.calls[-1][0].abs().sum()) == 0.0
        assert eng.kinds == (["recompute"] * 2 if drop else ["kept"] * 2)


def test_inference_only_models_refuse_training_mode():
    from nabladft_b200 import spk
    from nabladft_b200.qhnet import QHNet

    orb = {1: [0, 0, 1], 6: [0, 0, 0, 1, 1, 2], 7: [0, 0, 0, 1, 1, 2], 8: [0, 0, 0, 1, 1, 2], 9: [0, 0, 0, 1, 1, 2], 16: [0, 0, 0, 0, 1, 1, 1, 2],
           17: [0, 0, 0, 0, 1, 1, 1, 2], 35: [0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2]}
    net = QHNet(sh_lmax=4, hidden_size=128, bottle_hidden_size=32, num_gnn_layers=5, max_radius=12, num_nodes=83, radius_embed_dim=32, orbitals=orb).train()

    class D:
        pos = torch.zeros(2, 3)

    with pytest.raises(NotImplementedError):
        net(D())
    from nabladft_b200._lib import NablaB200Error

    with pytest.raises(NablaB200Error):  # eval mode on CPU tensors: no CPU fallback
        net.eval()(D())


def test_gemnet_oc_host_mirror_layout_state_dict_and_refusals():
    """nabladft_b200/gemnet_oc.py: canonical-layout name lists in step with the header enums, struct layout, yaml instantiation with the
    reference's 429 state-dict names / shapes (strict load of an oracle state dict), export sizes, and the loud refusals."""
    import yaml

    from nabladft_b200 import gemnet_oc as G
    from nabladft_b200._lib import GemNetOCWeights, NablaB200Error
    from oracle.gemnet_oc import GemNetOCOracle

    hdr = open(os.path.join(ROOT, "include", "nabla_b200.h")).read()
    for prefix, names in (("G", G.G_NAMES), ("I", G.I_NAMES), ("O", G.O_NAMES), ("S", G.S_NAMES), ("SO", G.SO_NAMES), ("C", G.C_NAMES)):
        assert G.header_enum_names(hdr, prefix) == names, prefix
    body = hdr[hdr.index("typedef struct nb200_gemnet_oc_weights {"):hdr.index("} nb200_gemnet_oc_weights;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S).split("{", 1)[1]
    names = []
    for decl in body.split(";"):
        decl = re.sub(r"^(const\s+)?(int32_t|int64_t|float)\s*\*?", "", decl.strip())
        names += [n.strip().lstrip("*").strip() for n in decl.split(",") if n.strip()]
    assert names == [f[0] for f in GemNetOCWeights._fields_]
    assert ctypes.sizeof(GemNetOCWeights) == 4 * 6 + 8 * 3

    cfg = yaml.safe_load(open(os.path.join(ROOT, "config", "model", "gemnet-oc-b200.yaml")))["net"]
    assert cfg.pop("_target_") == "nabladft_b200.gemnet_oc.GemNetOC"
    net = G.GemNetOC(**cfg).eval()
    ref_sd = GemNetOCOracle().state_dict()  # names and shapes pinned to the reference's classes (tests/test_oracle.py)
    sd = net.state_dict()
    assert len(sd) == 429 and {k: tuple(v.shape) for k, v in sd.items()} == {k: tuple(v.shape) for k, v in ref_sd.items()}
    net.load_state_dict(ref_sd, strict=True)
    assert net.num_params == 37815873
    buf, offs, scales = net.export(torch.device("cpu"))
    assert len(offs) == len(G.G_NAMES) + 4 * len(G.I_NAMES) + 5 * len(G.O_NAMES) and len(scales) == 4 * len(G.S_NAMES) + 5 * len(G.SO_NAMES)
    assert all(o % 64 == 0 for o in offs) and offs == sorted(offs) and buf.numel() > 37_000_000
    assert all(s == 1.0 for s in scales)  # unfitted factors (0) are the identity, scale_factor.py:77,148

    with pytest.raises(NablaB200Error):  # another size: outside the compiled path, refused at construction
        G.GemNetOC(**{**cfg, "emb_size_edge": 256})
    with pytest.raises(NablaB200Error):
        G.GemNetOC(**{**cfg, "direct_forces": False})

    class D:
        z, pos, batch = torch.ones(3, dtype=torch.long), torch.zeros(3, 3), torch.zeros(3, dtype=torch.long)

    with pytest.raises(NablaB200Error):  # CPU tensors: no CPU fallback
        with torch.no_grad():
            net(D())
    with pytest.raises(NablaB200Error):  # training mode: not built for this model
        net.train()(D())
