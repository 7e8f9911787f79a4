"""The run path against vectors produced by the reference's OWN code (tests/golden/make_run_reference_golden.py ran the
unmodified src/yacht/hypothesis_recovery_src.py + utils.py with stand-ins for the absent sourmash package / CLI).

CPU part: pins oracle/run_oracle.py (the restatement the other run-path tests check the GPU against).
GPU part: the C-ABI calls (K5 exclusive hashes, K6 statistics) and the drop-in hypothesis_recovery() against the same
vectors.  Integers bit-exact; floats within 1e-9 relative (the bar of tests/test_run_parity_gpu.py).
"""
import importlib.util
import os

import numpy as np
import pytest

from oracle import run_oracle as ro

GOLD = os.path.join(os.path.dirname(__file__), "golden")
REL_TOL = 1e-9


@pytest.fixture(scope="module")
def gold():
    return _generator().load(os.path.join(GOLD, "run_reference_golden.npz"))     # inputs re-made from their seeds


def _generator():
    spec = importlib.util.spec_from_file_location("make_run_reference_golden", os.path.join(GOLD, "make_run_reference_golden.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)          # importing it touches neither /root/reference nor sourmash
    return mod


def _variants(z, meta):
    for case in meta["cases_a"]:
        c = case["id"]
        for v in range(case["variants"]):
            yield c, v, z[f"a{c}_hashes"], z[f"a{c}_offsets"], z[f"a{c}_sample"], z[f"a{c}_mask{v}"], z[f"a{c}_info{v}"]


def test_fixture_shape(gold):
    z, meta = gold
    assert len(meta["cases_a"]) == 50 and len(meta["cases_b"]) == 6
    assert sum(c["variants"] for c in meta["cases_a"]) == 200
    assert z["hyp_in"].shape[0] == z["hyp_out"].shape[0] == 24340


def test_oracle_exclusive_counts_match_reference(gold):
    z, meta = gold
    checked = 0
    for c, v, hashes, offsets, sample, mask, info in _variants(z, meta):
        got = ro.exclusive_counts(hashes, offsets, sample, mask)
        ids = np.flatnonzero(mask)
        assert np.array_equal(got["n_exclusive"][ids], info[:, 0]), (c, v)
        assert np.array_equal(got["n_match"][ids], info[:, 1]), (c, v)
        assert np.array_equal(got["n_overlap"], z[f"a{c}_overlap"]), (c, v)
        checked += len(ids)
    assert checked > 2000


def test_oracle_single_hyp_test_matches_reference(gold):
    z, _ = gold
    hin, hout = z["hyp_in"], z["hyp_out"]
    step = 7                       # every 7th row: ~3,500 scipy evaluations, the rest are covered on the GPU side
    for i in range(0, hin.shape[0], step):
        ne, nm, k, sig, ani, cov = hin[i]
        cov = int(cov) if cov == 1 else float(cov)
        got = ro.single_hyp_test((int(ne), int(nm)), int(k), float(sig), float(ani), cov)
        exp = hout[i]
        assert bool(got[0]) == bool(exp[0]) and got[2:5] == tuple(int(x) for x in exp[2:5]) and got[5] == exp[5], (hin[i], got, exp)
        for a, b in ((got[1], exp[1]), (got[6], exp[6]), (got[7], exp[7])):
            assert ro.float_close(a, b, 1e-12), (hin[i], got, exp)


@pytest.mark.gpu
def test_gpu_exclusive_hashes_match_reference(gpu_ctx, gold):
    z, meta = gold
    loaded = None
    for c, v, hashes, offsets, sample, mask, info in _variants(z, meta):
        if loaded != c:
            gpu_ctx.load_sketches(hashes, offsets)
            loaded = c
        got = gpu_ctx.exclusive_hashes(sample, mask)
        ids = np.flatnonzero(mask)
        assert np.array_equal(got["n_exclusive"][ids].astype(np.int64), info[:, 0]), (c, v)
        assert np.array_equal(got["n_match"][ids].astype(np.int64), info[:, 1]), (c, v)
        assert np.array_equal(got["n_overlap"].astype(np.int64), z[f"a{c}_overlap"]), (c, v)
        if v == 0:                 # the call `yacht run` makes: no mask, nontrivial = overlap > 0
            got0 = gpu_ctx.exclusive_hashes(sample)
            assert np.array_equal(got0["nontrivial"].astype(np.uint8), mask), c
            assert np.array_equal(got0["n_exclusive"][ids].astype(np.int64), info[:, 0]), c
            assert np.array_equal(got0["n_match"][ids].astype(np.int64), info[:, 1]), c


@pytest.mark.gpu
def test_gpu_hyp_test_matches_reference(gpu_ctx, gold):
    z, meta = gold
    hin, hout = z["hyp_in"], z["hyp_out"]
    covs = [float(c) for c in meta["covs"]]
    total = 0
    for k, sig, ani in meta["hyp_grid"]:
        sel = np.flatnonzero((hin[:, 2] == k) & (hin[:, 3] == sig) & (hin[:, 4] == ani))
        rows_in, rows_out = hin[sel], hout[sel]
        # generator order: for each (ne, nm): for each cov
        assert rows_in.shape[0] % len(covs) == 0
        ne = rows_in[::len(covs), 0].astype(np.int64)
        nm = rows_in[::len(covs), 1].astype(np.int64)
        got = gpu_ctx.hyp_test(ne, nm, int(k), float(sig), float(ani), covs)
        exp = rows_out.reshape(len(ne), len(covs), 8)
        for r in range(len(ne)):
            for ci in range(len(covs)):
                g, e = got[ci, r], exp[r, ci]
                ctxt = f"ne={ne[r]} nm={nm[r]} k={k} sig={sig} ani={ani} cov={covs[ci]}: got {g} exp {e}"
                assert bool(g["in_sample_est"]) == bool(e[0]), ctxt
                assert int(g["num_exclusive_kmers"]) == int(e[2]), ctxt
                assert int(g["num_exclusive_kmers_coverage"]) == int(e[3]), ctxt
                assert int(g["num_matches"]) == int(e[4]), ctxt
                assert float(g["acceptance_threshold_with_coverage"]) == e[5], ctxt
                assert ro.float_close(float(g["p_val"]), e[1], REL_TOL), ctxt
                assert ro.float_close(float(g["actual_confidence_with_coverage"]), e[6], REL_TOL), ctxt
                assert ro.float_close(float(g["alt_confidence_mut_rate_with_coverage"]), e[7], REL_TOL), ctxt
                total += 1
    assert total == hin.shape[0]


@pytest.mark.gpu
def test_gpu_hypothesis_recovery_frames_match_reference(gold, tmp_path):
    """The drop-in hypothesis_recovery() on the same files the reference's hypothesis_recovery() was given."""
    from yacht_b200 import hypothesis_recovery_src as hr
    from yacht_b200 import sigio
    z, meta = gold
    gen = _generator()
    float_cols = ("p_vals", "acceptance_threshold_with_coverage", "actual_confidence_with_coverage",
                  "alt_confidence_mut_rate_with_coverage")
    for case in meta["cases_b"]:
        c = case["id"]
        offsets = z[f"b{c}_offsets"]
        hashes = z[f"b{c}_hashes"]
        sketches = [hashes[int(offsets[g]):int(offsets[g + 1])] for g in range(len(offsets) - 1)]
        root = str(tmp_path / f"b{c}")
        manifest = gen.write_db(root, sketches, case["ksize"], extra_ksize=case["extra_ksize"], seed=case["seed"])
        sdir = tmp_path / f"b{c}_sample"
        sdir.mkdir()
        sample_file = str(sdir / "sample.sig.zip")
        gen.write_sample_zip(sample_file, "sample", case["ksize"], z[f"b{c}_sample"])
        sample_sig = sigio.load_signature_with_ksize(sample_file, case["ksize"])
        frames = hr.hypothesis_recovery(manifest.copy(), (sample_file, sample_sig), root, case["covs"], 1000, case["ksize"],
                                        case["significance"], case["ani"], 2)
        assert len(frames) == len(case["frames"])
        for fr, exp, exact in zip(frames, case["frames"], case["frames_exact"]):
            assert list(fr.columns) == exp["columns"], c
            assert len(fr) == len(exp["data"]), c
            for j, col in enumerate(exp["columns"]):
                want = [row[j] for row in exp["data"]]
                have = fr[col].tolist()
                if col in float_cols:
                    for a, b in zip(have, exact[col]):
                        assert ro.float_close(float(a), float(b), REL_TOL), (c, col, a, b)
                elif col == "in_sample_est":
                    assert [bool(x) for x in have] == [bool(x) for x in want], (c, col)
                else:
                    assert have == want, (c, col)
