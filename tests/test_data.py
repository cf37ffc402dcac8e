"""Data path (nabladft_b200/data.py): ASE-sqlite reader semantics, packed cache round trip, batch iterator, rank sharding."""
import json
import os
import sqlite3
import struct

import numpy as np
import pytest
import torch

from helpers import GOLDEN

from nabladft_b200.data import DeviceBatcher, PackedEnergyDataset, read_ase_energy_db


def _ase_bytes(d):
    """Writer for ASE's binary `data` container (the format the nablaDFT energy DBs use): arrays first, JSON index last."""
    body, meta = bytearray(8), {}
    for k, v in d.items():
        v = np.ascontiguousarray(v)
        while len(body) % 8:
            body.append(0)
        meta[k] = {"__ndarray__": [list(v.shape), str(v.dtype), len(body)]}
        body += v.tobytes()
    off = len(body)
    body += json.dumps(meta).encode()
    body[:8] = struct.pack("<q", off)
    return bytes(body)


def _write_db(path, fx, mols):
    con = sqlite3.connect(path)
    con.execute("create table systems (id integer primary key autoincrement, numbers blob, positions blob, natoms integer, data blob)")
    for m in mols:
        a, b = int(fx["ptr"][m]), int(fx["ptr"][m + 1])
        data = _ase_bytes({"energy": np.array([fx["energy"][m]]), "forces": fx["forces"][a:b]})
        con.execute("insert into systems (numbers, positions, natoms, data) values (?, ?, ?, ?)",
                    (fx["z"][a:b].astype(np.int32).tobytes(), fx["pos"][a:b].astype(np.float64).tobytes(), b - a, data))
    con.commit(); con.close()


@pytest.fixture()
def packed(tmp_path):
    fx = np.load(os.path.join(GOLDEN, "fixture_molecules.npz"))
    mols = list(range(37))
    db = str(tmp_path / "mini.db")
    _write_db(db, fx, mols)
    return fx, mols, PackedEnergyDataset.from_ase_db(db), tmp_path


def test_reader_follows_reference_row_semantics(packed):
    fx, mols, ds, _ = packed
    n = int(fx["ptr"][len(mols)])
    assert len(ds) == len(mols) and ds.z.dtype == np.int32 and ds.pos.dtype == np.float32 and ds.forces.dtype == np.float32
    assert np.array_equal(ds.z, fx["z"][:n]) and np.array_equal(ds.ptr, fx["ptr"][:len(mols) + 1])
    assert np.array_equal(ds.pos, fx["pos"][:n].astype(np.float32))        # positions -> .float()  (pyg_datasets.py:106)
    assert np.array_equal(ds.forces, fx["forces"][:n].astype(np.float32))  # forces -> .float()     (pyg_datasets.py:108)
    assert np.array_equal(ds.energy, fx["energy"][:len(mols)].astype(np.float32))


def test_reader_on_the_reference_fixture_database():
    """The first rows of the reference's energy fixture DB, every ASE table kept (tests/golden/make_reference_samples.py)."""
    fx = np.load(os.path.join(GOLDEN, "fixture_molecules.npz"))
    d = read_ase_energy_db(os.path.join(GOLDEN, "energy_db_sample.db"))
    m = len(d["energy"])
    n = int(fx["ptr"][m])
    assert m == 10
    assert np.array_equal(d["z"], fx["z"][:n]) and np.array_equal(d["ptr"], fx["ptr"][:m + 1]) and np.array_equal(d["pos"], fx["pos"][:n].astype(np.float32))
    assert np.array_equal(d["forces"], fx["forces"][:n].astype(np.float32)) and np.array_equal(d["energy"], fx["energy"][:m].astype(np.float32))


def test_packed_cache_round_trip_is_memory_mapped(packed):
    _, _, ds, tmp = packed
    ds.save(str(tmp / "cache"))
    back = PackedEnergyDataset.load(str(tmp / "cache"))
    assert isinstance(back.pos, np.memmap)
    for f in PackedEnergyDataset.FIELDS:
        assert np.array_equal(np.asarray(getattr(back, f)), getattr(ds, f))
    m = back.molecule(5)
    assert len(m["z"]) == ds.n_atoms[5]


@pytest.mark.parametrize("shuffle", [False, True])
def test_batcher_covers_every_molecule_once_and_shards_are_disjoint(packed, shuffle):
    _, _, ds, _ = packed
    seen_all, steps = [], []
    for rank in range(3):
        it = DeviceBatcher(ds, batch_size=5, device="cpu", shuffle=shuffle, seed=7, rank=rank, world=3)
        it.set_epoch(2)
        seen = []
        for b in it:
            assert b.z.dtype == torch.int32 and b.pos.dtype == torch.float32 and b.mol_ptr.dtype == torch.int32
            assert int(b.mol_ptr[-1]) == b.z.shape[0] == b.pos.shape[0] == b.forces.shape[0] and b.energy.shape[0] == b.n_mol <= 10
            for k, m in enumerate(b.index.tolist()):  # every molecule arrives intact
                a, e = int(b.mol_ptr[k]), int(b.mol_ptr[k + 1])
                mol = ds.molecule(m)
                assert np.array_equal(b.z[a:e].numpy(), mol["z"]) and np.array_equal(b.pos[a:e].numpy(), mol["pos"])
                assert np.array_equal(b.forces[a:e].numpy(), mol["forces"]) and float(b.energy[k]) == float(mol["energy"])
            seen += b.index.tolist()
            spk = b.as_spk(); pyg = b.as_pyg()
            assert spk["_idx_m"].shape[0] == b.z.shape[0] and int(spk["_n_atoms"].sum()) == b.z.shape[0] and pyg.ptr.dtype == torch.int64
        assert len(seen) == len(set(seen))
        seen_all.append(seen)
        steps.append((len(it), sum(1 for _ in it)))
    # every rank takes the SAME number of steps (one gradient all-reduce per step: unequal counts dead-lock NCCL at the end of an epoch)
    assert len(set(steps)) == 1 and steps[0][0] == steps[0][1] > 0, steps
    flat = sum(seen_all, [])
    assert sorted(flat) == list(range(len(ds)))                      # ranks partition the epoch
    loads = [int(ds.n_atoms[s].sum()) for s in seen_all]
    assert max(loads) - min(loads) <= 2 * int(ds.n_atoms.max())      # atom-balanced shards
    if shuffle:
        again = DeviceBatcher(ds, batch_size=5, device="cpu", shuffle=True, seed=7, rank=0, world=3)
        again.set_epoch(2)
        assert sum((b.index.tolist() for b in again), []) == seen_all[0]   # deterministic in (seed, epoch)
        again.set_epoch(3)
        assert sum((b.index.tolist() for b in again), []) != seen_all[0]


@pytest.mark.parametrize("drop_last", [False, True])
def test_batcher_equal_steps_per_rank_with_unequal_molecule_sizes(drop_last):
    """Atom-balanced shards of a dataset whose molecules differ 10x in size hold very different molecule counts per rank; the
    number of batches per epoch must still agree (ADVICE r1: a rank with more batches blocks forever in the gradient all-reduce)."""
    rng = np.random.default_rng(0)
    n_atoms = np.concatenate([np.full(40, 3), np.full(12, 30)]).astype(np.int64)
    ptr = np.zeros(len(n_atoms) + 1, dtype=np.int64); np.cumsum(n_atoms, out=ptr[1:])
    tot = int(ptr[-1])
    ds = PackedEnergyDataset(z=rng.integers(1, 9, tot).astype(np.int32), pos=rng.normal(size=(tot, 3)).astype(np.float32),
                             forces=np.zeros((tot, 3), np.float32), energy=np.zeros(len(n_atoms), np.float32), ptr=ptr)
    for world in (2, 3):
        lens, seen = [], []
        for rank in range(world):
            it = DeviceBatcher(ds, batch_size=4, device="cpu", shuffle=False, drop_last=drop_last, rank=rank, world=world)
            got = [b.index.tolist() for b in it]
            lens.append((len(it), len(got)))
            seen += sum(got, [])
        assert len(set(lens)) == 1 and lens[0][0] == lens[0][1] > 0, (world, lens)
        assert sorted(seen) == list(range(len(n_atoms)))


def _write_hdb(path, mats, zs, rs):
    con = sqlite3.connect(path)
    con.execute("create table data (id integer not null primary key, Z blob, R blob, E float, F blob, H blob, S blob, C blob)")
    con.execute("create table metadata (id integer primary key, N integer)")
    con.execute("create table dataset_ids (id integer not null primary key, MOSES_ID int, CONFORMER_ID int)")
    con.execute("create table basisset (Z integer not null primary key, orbitals blob)")
    for i, (h, z, r) in enumerate(zip(mats, zs, rs)):
        con.execute("insert into data values (?, ?, ?, ?, ?, ?, ?, ?)", (i, z.astype(np.int32).tobytes(), r.astype(np.float32).tobytes(), -1.5 * i,
                                                                        (0.1 * r).astype(np.float32).tobytes(), h.astype(np.float32).tobytes(),
                                                                        np.eye(len(h), dtype=np.float32).tobytes(), None))
        con.execute("insert into dataset_ids values (?, ?, ?)", (i, 1000 + i, i % 3))
    con.execute("insert into metadata values (0, ?)", (len(mats),))
    con.execute("insert into basisset values (1, ?)", (np.array([0, 0, 1], dtype=np.int32).tobytes(),))
    con.commit(); con.close()


def test_hamiltonian_db_reader_and_packed_batches(tmp_path):
    from nabladft_b200.data import PackedHamiltonianDataset, read_hamiltonian_db
    from nabladft_b200.losses import HamiltonianLoss

    rng = np.random.default_rng(0)
    sizes, norbs = [3, 5, 4], [7, 12, 9]
    zs = [rng.integers(1, 9, n) for n in sizes]
    rs = [rng.standard_normal((n, 3)) for n in sizes]
    mats = [rng.standard_normal((k, k)) for k in norbs]
    db = str(tmp_path / "h.db")
    _write_hdb(db, mats, zs, rs)
    a = read_hamiltonian_db(db, include_overlap=True)
    assert a["norb"].tolist() == norbs and a["ptr"].tolist() == [0, 3, 8, 12] and a["h_off"].tolist() == [0, 49, 193, 274]
    assert np.array_equal(a["pos"], np.concatenate(rs).astype(np.float32)) and a["energy"].tolist() == [0.0, -1.5, -3.0]
    assert a["moses_id"].tolist() == [1000, 1001, 1002] and a["basis"][1].tolist() == [0, 0, 1] and a["S"].shape == a["H"].shape
    ds = PackedHamiltonianDataset.from_db(db)
    assert np.array_equal(ds.hamiltonian(1), mats[1].astype(np.float32))
    d, targets = ds.batch([2, 0], device="cpu")
    assert d.ptr.tolist() == [0, 4, 7] and d.batch.tolist() == [0] * 4 + [1] * 3 and d.z.dtype == torch.int64
    assert [tuple(t.shape) for t in targets] == [(9, 9), (7, 7)] and np.array_equal(targets[1].numpy(), mats[0].astype(np.float32))
    assert float(HamiltonianLoss.packed(targets, targets)) == 0.0


def test_hamiltonian_reader_on_the_reference_fixture_database():
    """The reference's Hamiltonian fixture DB cut to its first 4 molecules, each to its first 4 atoms and the principal sub-blocks of H and S
    over their orbitals (tests/golden/make_reference_samples.py): the reader decodes its real layout and units."""
    from nabladft_b200.data import read_hamiltonian_db

    a = read_hamiltonian_db(os.path.join(GOLDEN, "hamiltonian_db_sample.db"), include_overlap=True)
    assert len(a["energy"]) == 4 and a["ptr"].tolist() == [0, 4, 8, 12, 16] and a["norb"].tolist() == [56] * 4  # 4 heavy atoms of 14 orbitals
    assert a["moses_id"].tolist() == [1292954, 513946, 863412, 292539] and abs(float(a["energy"][0]) + 1711.5248) < 1e-3
    for m in range(4):
        no, o = int(a["norb"][m]), int(a["h_off"][m])
        for mat in (a["H"], a["S"]):
            h = mat[o: o + no * no].reshape(no, no)
            assert np.abs(h - h.T).max() < 1e-5                                                    # Fock and overlap matrices are symmetric
        p = a["pos"][a["ptr"][m]: a["ptr"][m + 1]]
        assert 1.5 < np.min([np.linalg.norm(p[i] - p[j]) for i in range(len(p)) for j in range(i)]) < 2.9  # bohr, not angstrom
        # orbitals per element from the basis table reproduce Norb (def2-SVP: 2l+1 per shell)
        assert sum(int((2 * a["basis"][int(zz)] + 1).sum()) for zz in a["z"][a["ptr"][m]: a["ptr"][m + 1]]) == no
