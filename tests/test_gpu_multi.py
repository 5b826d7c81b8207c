"""Several GPUs in one box (marker `multigpu`: skipped with fewer than 2 devices; the argument checks run on one).

(1) ONE process driving N devices through the C ABI (ihtb_mgeno / ihtb_mfit / ihtb_mcv_run): the SNP-sharded fit must
    reproduce the single-GPU fit (same support, iterations, backtracks; beta to 1e-9 -- the all-reduce adds the shard
    partials in rank order, so only the association of the X*beta sums differs), and the farmed CV grid must equal the
    single-GPU grid bit for bit (replicas, no data-path collective).
(2) one process per GPU (torchrun + NCCL rendezvous + CUDA IPC peer memory): scripts/check_sharded.py as a subprocess."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import mendeliht_jl_b200 as m
from mendeliht_jl_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NGPU = min(m.device_count(), int(os.environ.get("IHTB_TEST_NGPU", "8"))) if m.device_count() else 0
Multi = m.B200MultiSnpLinAlg


def _same(res, ref, rtol=1e-9):
    assert res.iter == ref.iter
    assert np.array_equal(np.flatnonzero(res.beta), np.flatnonzero(ref.beta))
    assert [t[1] for t in res.trace] == [t[1] for t in ref.trace]
    np.testing.assert_allclose(res.beta, ref.beta, rtol=rtol, atol=1e-12)
    np.testing.assert_allclose(res.c, ref.c, rtol=rtol, atol=1e-12)
    assert abs(res.logl - ref.logl) <= rtol * abs(ref.logl)
    np.testing.assert_allclose([t[0] for t in res.trace], [t[0] for t in ref.trace], rtol=rtol)


@pytest.mark.multigpu
@pytest.mark.parametrize("d,l,n,p,k,ncov,miss", [("Normal", "IdentityLink", 5000, 20001, 8, 2, 0.0),
                                                 ("Bernoulli", "LogitLink", 6000, 16000, 6, 0, 0.001),
                                                 ("Poisson", "LogLink", 4000, 12000, 6, 1, 0.0),
                                                 # n > 262144: the X*beta all-reduce takes the two-phase path
                                                 ("Normal", "IdentityLink", 300001, 4000, 6, 1, 0.0)])
def test_one_process_sharded_fit_matches_single_gpu(d, l, n, p, k, ncov, miss):
    seed = 11 + n
    y, z, *_ = synth.simulate_response(seed, n, p, k, d, n_cov=ncov, missing_rate=miss)
    gm = Multi.synthetic(n, p, seed, miss, ngpu=NGPU, mode=Multi.SHARD)
    g1 = m.B200SnpLinAlg.synthetic(n, p, seed, miss)
    for mode in (m.SWEEP_FAST, m.SWEEP_EXACT):
        res = m.fit_iht(y, gm, z, k=k + 2, d=d, l=l, sweep_mode=mode)
        ref = m.fit_iht(y, g1, z, k=k + 2, d=d, l=l, sweep_mode=mode)
        _same(res, ref)
    gm.close(); g1.close()


@pytest.mark.multigpu
def test_one_process_sharded_options_match_single_gpu():
    """weights, init_beta, groups (scalar and per-group k, groups straddling the shard boundary) and debias."""
    n, p, k = 4000, 16000, 6
    y, z, *_ = synth.simulate_response(55, n, p, k, "Normal", n_cov=1)
    bed = synth.packed_columns(55, n, np.arange(p))
    gm = Multi.from_bed_columns(bed, n, ngpu=NGPU, mode=Multi.SHARD)          # host .bed bytes split over the devices
    g1 = m.B200SnpLinAlg.from_bed_columns(bed, n)
    w = m.maf_weights(g1, max_weight=4.0)
    _same(m.fit_iht(y, gm, z, k=k + 2, weight=w), m.fit_iht(y, g1, z, k=k + 2, weight=w))
    _same(m.fit_iht(y, gm, z, k=k + 2, init_beta=True), m.fit_iht(y, g1, z, k=k + 2, init_beta=True))
    blocks = np.arange(p) // 333 + 1
    for kw in ({"k": 2, "J": 4}, {"k": [2] * int(blocks.max()), "J": 3}):
        _same(m.fit_iht(y, gm, z, group=blocks, **kw), m.fit_iht(y, g1, z, group=blocks, **kw))
    yb, zb, *_ = synth.simulate_response(56, n, p, k, "Bernoulli", geno_seed=55)
    _same(m.fit_iht(yb, gm, zb, k=k + 1, d="Bernoulli", l="LogitLink", debias=True),
          m.fit_iht(yb, g1, zb, k=k + 1, d="Bernoulli", l="LogitLink", debias=True), rtol=1e-8)
    # a part is an ordinary single-device operator over its column block
    part = gm.part(NGPU - 1)
    assert np.array_equal(part.packed(), bed[part.j0:part.j0 + part.p])
    gm.close(); g1.close()


@pytest.mark.multigpu
@pytest.mark.parametrize("n,p,r,k", [(1200, 2500, 2, 8), (1003, 1500, 5, 10), (4000, 9000, 3, 12)])
def test_one_process_sharded_multivariate_fit_matches_single_gpu(n, p, r, k):
    """MvNormal fit (mIHTVariable) with the SNP columns split over the devices: n x r products all-reduced, exact
    gradient entries and candidate columns exchanged; FAST, EXACT and PAIR sweeps."""
    rng = np.random.default_rng(40 + r)
    bed = synth.packed_columns(40 + r, n, np.arange(p))
    idx = np.sort(rng.permutation(p)[:k])
    B = np.zeros((r, k))
    for c in range(k):
        B[rng.integers(0, r), c] = rng.normal() * 0.8
    Y = B @ synth.standardized_columns(40 + r, n, idx).T + rng.normal(size=(r, n))
    Z = np.vstack([np.ones(n), rng.normal(size=n)])
    gm = Multi.from_bed_columns(bed, n, ngpu=NGPU, mode=Multi.SHARD)
    g1 = m.B200SnpLinAlg.from_bed_columns(bed, n)
    for mode in (m.SWEEP_FAST, m.SWEEP_EXACT, m.SWEEP_PAIR):
        res = m.fit_iht(Y, gm, Z, k=k + 2, sweep_mode=mode)
        ref = m.fit_iht(Y, g1, Z, k=k + 2, sweep_mode=mode)
        assert res.iter == ref.iter and np.array_equal(res.beta != 0, ref.beta != 0)
        assert [t[1] for t in res.trace] == [t[1] for t in ref.trace]
        np.testing.assert_allclose(res.beta, ref.beta, rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(res.c, ref.c, rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(res.Sigma, ref.Sigma, rtol=1e-8, atol=1e-12)
        assert abs(res.logl - ref.logl) <= 1e-9 * abs(ref.logl)
    # init_beta (initialize_beta!, src/multivariate.jl:519-558): per-shard regressions, intercept sums all-reduced, the
    # ranks' top-k entries of the initial B all-gathered
    res = m.fit_iht(Y, gm, Z, k=k + 2, init_beta=True)
    ref = m.fit_iht(Y, g1, Z, k=k + 2, init_beta=True)
    assert res.iter == ref.iter and np.array_equal(res.beta != 0, ref.beta != 0)
    np.testing.assert_allclose(res.beta, ref.beta, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(res.c, ref.c, rtol=1e-9, atol=1e-12)
    assert abs(res.logl - ref.logl) <= 1e-9 * abs(ref.logl)
    gm.close(); g1.close()


@pytest.mark.multigpu
def test_one_process_cv_farm_matches_single_gpu():
    n, p, q = 6000, 20000, 3
    path = [1, 2, 4, 6, 9]
    y, z, *_ = synth.simulate_response(2025, n, p, 6, "Poisson", geno_seed=2025)
    folds = synth.folds_for(2025, n, q)
    gm = Multi.synthetic(n, p, 2025, 0.0, ngpu=NGPU, mode=Multi.REPLICATE)
    g1 = m.B200SnpLinAlg.synthetic(n, p, 2025)
    mses, iters = m.cv_run(y, gm, z, folds, q, path, d="Poisson", l="LogLink")
    rm, ri = m.cv_run(y, g1, z, folds, q, path, d="Poisson", l="LogLink")
    assert np.array_equal(iters, ri) and np.array_equal(mses, rm)
    assert m.cv_run.last_busy_seconds.shape == (NGPU,) and np.all(m.cv_run.last_busy_seconds > 0)
    with pytest.raises(m.IHTBError):                 # a fit over replicas is a usage error, not a silent single-GPU fit
        m.fit_iht(y, gm, z, k=3, d="Poisson", l="LogLink")
    gm.close(); g1.close()


def test_multi_handle_argument_errors():
    with pytest.raises(m.IHTBError):
        Multi.synthetic(100, 50, 1, 0.0, ngpu=m.device_count() + 1)
    with pytest.raises(m.IHTBError):
        Multi.synthetic(100, 50, 1, 0.0, ngpu=2, devices=[0, 0])


@pytest.mark.multigpu
def test_one_process_per_gpu_sharded_fit_torchrun():
    """The multi-process form (what bench.py --gpus N runs): NCCL rendezvous, CUDA IPC peer memory."""
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={min(NGPU, 2)}",
           "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.join(ROOT, "scripts", "check_sharded.py")]
    env = dict(os.environ, CHECK_SHARDED_SKIP_FULL="1")
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "same=False" not in out.stdout
