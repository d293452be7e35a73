"""CPU suite: argument checks of the multi-response Python layer and the cv-multi file loader (no device needed)."""
import numpy as np
import pytest


@pytest.fixture(scope="module")
def pb(built):
    import pareben_b200 as pb
    return pb


def test_shape_mismatch_raises(pb):
    X = np.zeros((10, 3))
    with pytest.raises(ValueError, match="n x T"):
        pb.CrossValidateMulti(X, np.zeros((9, 2)), 2)
    with pytest.raises(ValueError, match="n x T"):
        pb.CrossValidateMulti(X, np.zeros(10), 2)                      # a vector is not a response matrix
    with pytest.raises(ValueError, match="n x T"):
        pb.CrossValidateMulti(X, np.zeros((10, 0)), 2)                 # T < 1
    with pytest.raises(ValueError, match="n x T"):
        pb.cv_grid_multi(X, np.zeros((11, 2)), np.ones(10), 2, np.ones((2, 3)), np.ones((2, 3)))
    with pytest.raises(ValueError, match=r"\(2, n_grid\)"):
        pb.cv_grid_multi(X, np.zeros((10, 2)), np.ones(10), 2, np.ones((3, 3)), np.ones((3, 3)))
    with pytest.raises(ValueError, match="at least one response"):
        pb.Problem(X, np.zeros((10, 0)))


def test_non_finite_names_its_column(pb):
    X = np.zeros((10, 3))
    Y = np.ones((10, 4))
    Y[3, 2] = np.nan
    with pytest.raises(ValueError, match="column 2.*missing rows are not supported"):
        pb.CrossValidateMulti(X, Y, 2)
    Y[3, 2] = 1.0
    Y[0, 1] = np.inf
    with pytest.raises(ValueError, match="column 1"):
        pb.CrossValidateMulti(X, Y, 2, search="local")


def _write(path, lines):
    path.write_text("\n".join(lines) + "\n")
    return str(path)


def test_loader_joins_phenotypes_on_ids(tmp_path):
    from pareben_b200 import io as pio
    geno = _write(tmp_path / "geno.txt", ["id\tm1\tm2", "a\t0\t1", "b\t1\t1", "c\t-1\t0"])
    p1 = _write(tmp_path / "p1.txt", ["c 3.0", "a 1.0", "b 2.0"])
    p2 = _write(tmp_path / "p2.txt", ["a 10.0", "b 20.0", "c 30.0"])              # same ids, another order
    X, Y = pio.load_problem_multi(geno, [p1, p2])
    assert np.array_equal(Y, [[3.0, 30.0], [1.0, 10.0], [2.0, 20.0]])             # rows in the order of the first file
    assert np.array_equal(X, [[-1, 0], [0, 1], [1, 1]])
    bad = _write(tmp_path / "p3.txt", ["a 1.0", "b 2.0", "d 4.0"])
    with pytest.raises(ValueError, match="sample ids differ"):
        pio.load_problem_multi(geno, [p1, bad])
    short = _write(tmp_path / "p4.txt", ["a 1.0", "b 2.0"])
    with pytest.raises(ValueError, match="sample ids differ"):
        pio.load_problem_multi(geno, [p1, short])


def test_loader_matrix_file(tmp_path):
    from pareben_b200 import io as pio
    X = np.arange(12.0).reshape(4, 3)
    Y = np.arange(8.0).reshape(4, 2)
    np.save(tmp_path / "X.npy", X)
    np.save(tmp_path / "Y.npy", Y)
    X2, Y2 = pio.load_problem_multi(str(tmp_path / "X.npy"), [str(tmp_path / "Y.npy")])
    assert np.array_equal(X2, X) and np.array_equal(Y2, Y)
    np.save(tmp_path / "y0.npy", Y[:, 0])
    np.save(tmp_path / "y1.npy", Y[:, 1])
    _X3, Y3 = pio.load_problem_multi(str(tmp_path / "X.npy"), [str(tmp_path / "y0.npy"), str(tmp_path / "y1.npy")])
    assert np.array_equal(Y3, Y)


def test_cli_cv_multi_parses_repeated_targets(tmp_path, monkeypatch):
    """The subcommand reads every --target and hands one n x T matrix to CrossValidateMulti."""
    from pareben_b200 import cli
    from pareben_b200 import cross_validate as cv
    seen = {}

    def fake(X, Y, nFolds, foldId=0, Epis="no", prior="gaussian", search="global", **kw):
        seen["shape"] = Y.shape
        return [{"lambda.optimal": 1.0, "alpha.optimal": 0.5, "Results.Summary": {"alpha": [0.5], "lambda": [1.0], "SE": [0.0], "MSE": [2.0]}}
                for _ in range(Y.shape[1])]

    monkeypatch.setattr(cv, "CrossValidateMulti", fake)
    geno = _write(tmp_path / "geno.txt", ["id\tm1\tm2"] + [f"s{i}\t{i % 3 - 1}\t{i % 2}" for i in range(6)])
    p1 = _write(tmp_path / "p1.txt", [f"s{i} {i}.5" for i in range(6)])
    p2 = _write(tmp_path / "p2.txt", [f"s{i} {2 * i}.5" for i in reversed(range(6))])
    out = tmp_path / "out.json"
    assert cli.main(["cv-multi", "--basis", geno, "--target", p1, "--target", p2, "--nfolds", "2", "--out", str(out)]) == 0
    import json
    res = json.loads(out.read_text())
    assert seen["shape"] == (6, 2) and isinstance(res, list) and len(res) == 2 and res[1]["lambda.optimal"] == 1.0
