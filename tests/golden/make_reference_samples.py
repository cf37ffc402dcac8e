"""Small samples of the reference checkout's data fixtures, for tests that must run without that checkout.

    python tests/golden/make_reference_samples.py <reference checkout>

writes
  energy_db_sample.db          the first ENERGY_ROWS rows of tests/data/raw/test_database.db (ASE-sqlite v9), every table
                               kept, the other rows deleted
  hamiltonian_db_sample.db     tests/data/raw/test_hamiltonian_database.db cut to its first HAM_ROWS molecules, each cut to its
                               first HAM_ATOMS atoms: Z / R / F rows of those atoms and the principal sub-blocks of H and S over
                               their orbitals (orbitals are stored atom by atom), metadata N set to HAM_ROWS
  reference_model_configs.yaml config/model/{painn-oc,painn,schnet,qhnet,gemnet-oc}.yaml as parsed, one mapping per file name
"""
import os
import shutil
import sqlite3
import sys

import numpy as np
import yaml

HERE = os.path.dirname(os.path.abspath(__file__))
ENERGY_ROWS = 10
HAM_ROWS, HAM_ATOMS = 4, 4
MODEL_YAMLS = ("painn-oc.yaml", "painn.yaml", "schnet.yaml", "qhnet.yaml", "gemnet-oc.yaml")


def _copy(src, dst):
    if os.path.exists(dst):
        os.remove(dst)
    shutil.copyfile(src, dst)
    os.chmod(dst, 0o644)
    con = sqlite3.connect(dst)
    con.execute("pragma page_size = 1024")  # applied by the final vacuum: the many empty tables and indices then take 1 KB each
    return con


def energy_sample(ref):
    con = _copy(os.path.join(ref, "tests", "data", "raw", "test_database.db"), os.path.join(HERE, "energy_db_sample.db"))
    for table in ("species", "keys", "text_key_values", "number_key_values", "systems"):
        con.execute(f"delete from {table} where id > ?", (ENERGY_ROWS,))
    con.execute("update sqlite_sequence set seq = ? where name = 'systems'", (ENERGY_ROWS,))
    con.commit()
    con.execute("vacuum")
    con.close()


def hamiltonian_sample(ref):
    con = _copy(os.path.join(ref, "tests", "data", "raw", "test_hamiltonian_database.db"), os.path.join(HERE, "hamiltonian_db_sample.db"))
    basis = {int(z): np.frombuffer(b, dtype=np.int32) for z, b in con.execute("select Z, orbitals from basisset")}
    con.execute("delete from data where id >= ?", (HAM_ROWS,))
    con.execute("delete from dataset_ids where id >= ?", (HAM_ROWS,))
    con.execute("update metadata set N = ? where id = 0", (HAM_ROWS,))
    for i, Zb, Rb, Fb, Hb, Sb in con.execute("select id, Z, R, F, H, S from data order by id").fetchall():
        z = np.frombuffer(Zb, dtype=np.int32)
        no = int(round((len(Hb) // 4) ** 0.5))
        k = sum(int((2 * basis[int(zz)] + 1).sum()) for zz in z[:HAM_ATOMS])
        sub = lambda b: np.frombuffer(b, dtype=np.float32).reshape(no, no)[:k, :k].copy().tobytes()
        con.execute("update data set Z = ?, R = ?, F = ?, H = ?, S = ? where id = ?",
                    (z[:HAM_ATOMS].tobytes(), Rb[: 12 * HAM_ATOMS], Fb[: 12 * HAM_ATOMS], sub(Hb), sub(Sb), i))
    con.commit()
    con.execute("vacuum")
    con.close()


def model_configs(ref):
    out = {fn: yaml.safe_load(open(os.path.join(ref, "config", "model", fn))) for fn in MODEL_YAMLS}
    with open(os.path.join(HERE, "reference_model_configs.yaml"), "w") as f:
        yaml.safe_dump(out, f, sort_keys=False)


if __name__ == "__main__":
    ref = sys.argv[1]
    energy_sample(ref)
    hamiltonian_sample(ref)
    model_configs(ref)
