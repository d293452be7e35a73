"""CPU suite: the file readers either side of the hot path (pareben_b200/io.py, rdata.py) and the command line's
argument handling.  The .rda reader reads the bundled inputs stored as R data files under tests/golden
(make_rda_golden.py); the text formats are exercised on files written here in the layout of the reference's own inputs
(genotype_full.txt, pheno_left.txt)."""
import os
import zipfile

import numpy as np
import pytest

from conftest import GOLDEN, golden


def _write_genotypes(path, ids, names, M):
    with open(path, "w") as f:
        f.write("SAMID\t" + "\t".join(names) + "\n")
        for s, row in zip(ids, M):
            f.write(s + "\t" + "\t".join(str(int(v)) for v in row) + "\n")


def test_genotype_and_phenotype_text_join(tmp_path):
    from pareben_b200 import io as pio
    rng = np.random.default_rng(3)
    ids = [f"{a:02d}_{b:02d}" for a in range(1, 4) for b in range(1, 6)]
    names = [f"{100 + j}_chrI_{100 + j}_A_T" for j in range(7)]
    M = rng.choice([-1, 1], size=(len(ids), 7))
    gpath = str(tmp_path / "genotype.txt")
    _write_genotypes(gpath, ids, names, M)
    keep = [ids[i] for i in (9, 2, 4, 13, 0)]                                   # phenotype order, a subset
    ppath = str(tmp_path / "pheno.txt")
    open(ppath, "w").write("".join(f"{s}\t{0.25 * i - 1:.6f}\n" for i, s in enumerate(keep)))
    got_ids, got_names, G = pio.read_genotype_text(gpath)
    assert G.dtype == np.int8 and np.array_equal(G, M) and list(got_ids) == ids and list(got_names) == names
    X, y = pio.load_problem(gpath, ppath)
    assert np.array_equal(X, M[[9, 2, 4, 13, 0]]) and np.allclose(y, 0.25 * np.arange(5) - 1)
    zpath = str(tmp_path / "genotype.zip")
    with zipfile.ZipFile(zpath, "w", zipfile.ZIP_DEFLATED) as z:
        z.write(gpath, "genotype_full.txt")
    Xz, yz = pio.load_problem(zpath, ppath)
    assert np.array_equal(Xz, X) and np.array_equal(yz, y)
    open(ppath, "a").write("99_99\t1.0\n")
    with pytest.raises(ValueError):
        pio.load_problem(gpath, ppath)
    open(gpath, "a").write("04_01\t" + "\t".join(["0.5"] * 7) + "\n")                 # not a genotype code
    with pytest.raises(ValueError):
        pio.read_genotype_text(gpath)
    assert pio.read_genotype_text(gpath, dtype=np.float64)[2][-1, 0] == 0.5


def test_rda_reader_against_bundled_inputs():
    from pareben_b200 import io as pio
    d = GOLDEN
    g = golden("inputs_bundled.npz")
    X = pio.read_matrix(os.path.join(d, "BASIS.rda"))
    y = pio.read_matrix(os.path.join(d, "y.rda"))
    assert X.shape == (1000, 481) and np.array_equal(X, g["BASIS"]) and np.array_equal(np.ravel(y), g["y"])
    Xb, yb = pio.load_problem(os.path.join(d, "BASISbinomial.rda"), os.path.join(d, "yBinomial.rda"))
    assert np.array_equal(Xb, g["BASISbinomial"]) and np.array_equal(yb, g["yBinomial"])


def test_cli_parses_and_needs_a_device(tmp_path, built):
    import pareben_b200 as pb
    from pareben_b200 import cli
    with pytest.raises(SystemExit):
        cli.main(["cv", "--basis", "x"])                                             # --target / --nfolds missing
    if pb.device_count() > 0:
        pytest.skip("a device is present")
    np.save(tmp_path / "X.npy", np.ones((8, 3))); np.save(tmp_path / "y.npy", np.arange(8.0))
    with pytest.raises(pb.ParebenError):                                            # no CPU fallback behind the command line either
        cli.main(["lambda-max", "--basis", str(tmp_path / "X.npy"), "--target", str(tmp_path / "y.npy")])
