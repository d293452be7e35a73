"""CPU suite: the host side of the batched final models (pareben_fit_batch, EBelasticNetMulti, the fit-multi command).

  * the weight table EBelasticNetMulti builds from a compact record equals _weight_table on the reference-layout table
    pareben_fit returns, for all four layouts, on synthetic records with zero betas and Epis main / pair mixes;
  * candidate_loci, the one place in Python that knows the candidate numbering, inverts it for every id;
  * fit-multi's argument handling, including a cv-multi JSON;
  * the new C entries are bound.
"""
import json

import numpy as np
import pytest

from record_layout import expand, keep_rows


@pytest.fixture(scope="module")
def pb(built):
    import pareben_b200 as pb
    return pb


def _record(rng, k, epis, gaussian, m):
    """A synthetic record: m distinct candidate ids in a random (Used) order, some betas exactly 0."""
    kc = (k + 1) * k // 2 if epis else k
    ids = rng.choice(kc, size=m, replace=False) + 1
    if epis and m >= 2:                            # make sure both main effects and pairs are present
        ids[0], ids[1] = rng.integers(1, k + 1), k + 1 + rng.integers(0, kc - k)
        ids = np.unique(ids)[rng.permutation(np.unique(ids).size)]
    m = ids.size
    beta = rng.normal(size=m) * (rng.random(m) > 0.3)
    var = rng.random(m) + 0.01
    return m, ids, beta, var


@pytest.mark.parametrize("gaussian", [True, False])
@pytest.mark.parametrize("epis", [False, True])
def test_record_weight_equals_reference_table_weight(pb, gaussian, epis):
    from pareben_b200.cross_validate import _record_weight, _weight_table
    rng = np.random.default_rng(3 + 2 * gaussian + epis)
    k, n = 12, 57
    for trial in range(40):
        m = int(rng.integers(0, 2 * k if (epis and not gaussian) else k))
        if trial == 0:
            m = 0
        if m:
            m, ids, beta, var = _record(rng, k, epis, gaussian, m)
        else:
            ids, beta, var = np.zeros(0, int), np.zeros(0), np.zeros(0)
        if trial == 1 and m:
            beta[:] = 0                            # every effect zero: the reference's one-row fallback
        me = 2 * k + 3
        cand = np.zeros(me, np.int32); cand[:m] = ids
        b = np.zeros(me); b[:m] = beta
        v = np.zeros(me); v[:m] = var
        table = expand(m, cand, b, v, k, epis, gaussian)
        want = _weight_table(table, keep_rows(table, epis, gaussian), epis, n)
        got = _record_weight(m, cand, b, v, epis, gaussian, k, n)
        assert np.array_equal(got, want, equal_nan=True), f"trial {trial}"


@pytest.mark.parametrize("k", [2, 3, 7, 50, 301])
def test_candidate_loci_inverts_the_enumeration(pb, k):
    ids, li, lj = list(range(k)), list(range(1, k + 1)), list(range(1, k + 1))
    for i in range(k - 1):
        for j in range(i + 1, k):
            ids.append(len(ids)); li.append(i + 1); lj.append(j + 1)
    gi, gj = pb.candidate_loci(np.array(ids), k)
    assert np.array_equal(gi, li) and np.array_equal(gj, lj)
    # one id at a time too (the scalar path of the same helper)
    for c in (0, k - 1, k, len(ids) - 1):
        assert (int(pb.candidate_loci(c, k)[0]), int(pb.candidate_loci(c, k)[1])) == (li[c], lj[c])


def _write(path, lines):
    path.write_text("\n".join(lines) + "\n")
    return str(path)


def _fake_multi(seen):
    def fake(X, Y, lam, alpha, Epis="no", prior="gaussian", device=None):
        seen.update(shape=Y.shape, lam=np.asarray(lam).tolist(), alpha=np.asarray(alpha).tolist(), epis=Epis, prior=prior)
        return [{"weight": np.zeros((1, 6)), "WaldScore": 1.0, "Intercept": 0.5, "residVar": 2.0, "lambda": float(lam[t]),
                 "alpha": float(alpha[t]), "status": 0} for t in range(Y.shape[1])]
    return fake


def test_cli_fit_multi_reads_a_cv_multi_json(pb, tmp_path, monkeypatch):
    from pareben_b200 import cli
    from pareben_b200 import cross_validate as cv
    seen = {}
    monkeypatch.setattr(cv, "EBelasticNetMulti", _fake_multi(seen))
    geno = _write(tmp_path / "geno.txt", ["id\tm1\tm2"] + [f"s{i}\t{i % 3 - 1}\t{i % 2}" for i in range(6)])
    p1 = _write(tmp_path / "p1.txt", [f"s{i} {i}.5" for i in range(6)])
    p2 = _write(tmp_path / "p2.txt", [f"s{i} {2 * i}.5" for i in reversed(range(6))])
    cvj = tmp_path / "cv.json"
    cvj.write_text(json.dumps([{"lambda.optimal": 0.25, "alpha.optimal": 0.5, "CrossValidation": []},
                               {"lambda.optimal": 0.125, "alpha.optimal": 0.75, "CrossValidation": []}]))
    out = tmp_path / "out.json"
    assert cli.main(["fit-multi", "--basis", geno, "--target", p1, "--target", p2, "--cv", str(cvj), "--epis", "yes",
                     "--out", str(out)]) == 0
    res = json.loads(out.read_text())
    assert seen == {"shape": (6, 2), "lam": [0.25, 0.125], "alpha": [0.5, 0.75], "epis": "yes", "prior": "gaussian"}
    assert isinstance(res, list) and len(res) == 2 and res[1]["lambda"] == 0.125 and res[0]["weight"] == [[0.0] * 6]


def test_cli_fit_multi_one_point_for_every_response(pb, tmp_path, monkeypatch):
    from pareben_b200 import cli
    from pareben_b200 import cross_validate as cv
    seen = {}
    monkeypatch.setattr(cv, "EBelasticNetMulti", _fake_multi(seen))
    np.save(tmp_path / "X.npy", np.arange(12.0).reshape(4, 3))
    np.save(tmp_path / "Y.npy", np.arange(12.0).reshape(4, 3))
    out = tmp_path / "out.json"
    assert cli.main(["fit-multi", "--basis", str(tmp_path / "X.npy"), "--target", str(tmp_path / "Y.npy"), "--lambda", "0.5",
                     "--alpha", "1", "--prior", "binomial", "--out", str(out)]) == 0
    assert seen["shape"] == (4, 3) and seen["lam"] == [0.5] * 3 and seen["alpha"] == [1.0] * 3 and seen["prior"] == "binomial"
    assert len(json.loads(out.read_text())) == 3


def test_cli_fit_multi_argument_errors(pb, tmp_path, monkeypatch):
    from pareben_b200 import cli
    from pareben_b200 import cross_validate as cv
    monkeypatch.setattr(cv, "EBelasticNetMulti", _fake_multi({}))
    np.save(tmp_path / "X.npy", np.arange(12.0).reshape(4, 3))
    np.save(tmp_path / "Y.npy", np.arange(8.0).reshape(4, 2))
    base = ["fit-multi", "--basis", str(tmp_path / "X.npy"), "--target", str(tmp_path / "Y.npy")]
    with pytest.raises(SystemExit, match="either --cv"):
        cli.main(base)                                                   # neither --cv nor --lambda/--alpha
    with pytest.raises(SystemExit, match="either --cv"):
        cli.main(base + ["--lambda", "1"])                               # --alpha missing
    cvj = tmp_path / "cv.json"
    cvj.write_text(json.dumps([{"lambda.optimal": 1.0, "alpha.optimal": 1.0}]))
    with pytest.raises(SystemExit, match="either --cv"):
        cli.main(base + ["--cv", str(cvj), "--lambda", "1", "--alpha", "1"])
    with pytest.raises(SystemExit, match="one entry per response"):
        cli.main(base + ["--cv", str(cvj)])                              # 1 entry, 2 responses


def test_ebelasticnet_multi_checks_arguments(pb):
    X = np.zeros((10, 3))
    with pytest.raises(ValueError, match="n x T"):
        pb.EBelasticNetMulti(X, np.zeros(10), 1.0, 1.0)
    with pytest.raises(ValueError, match="one entry per response"):
        pb.EBelasticNetMulti(X, np.zeros((10, 2)), [1.0, 2.0, 3.0], 1.0)


def test_new_entries_are_bound(pb):
    assert {"pareben_fit_batch", "pareben_max_effects"} <= set(pb._lib.SIGNATURES)
    assert len(pb._lib.SIGNATURES["pareben_fit_batch"][1]) == 14
