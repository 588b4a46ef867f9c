"""CPU: pins for N1 (CMA-ES).  Three layers:

1. oracle/cmaes_oracle.py (the restatement) == the reference's OWN objects (oracle/_ref/libcmaes_ref.so: the
   unmodified CmaEsSolverTorch.cpp + Controller.cpp compiled against pip-torch's libtorch) on identical seeds --
   samples and every state tensor BIT FOR BIT, generation after generation (both call the same ATen kernels);
2. the restatement == tests/golden/cmaes_ref.npz, minted from that library (tools/make_golden_cmaes.py), so the pin
   also holds where the reference's sources and the compiled library are absent;
3. the product (openkitchen_b200/cmaes.py: batched, binary64 partial sums) == the restatement to float32 rounding:
   the reference narrows its binary64 sums to float32 after every candidate, the product once (tolerances below)."""
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from openkitchen_b200.cmaes import CmaEs, PopulationController  # noqa: E402
from oracle.cmaes_oracle import (CmaEsOracle, CmaEsReference, controller_forward, have_ref,  # noqa: E402
                                 reference_controller_forward)

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cmaes_ref.npz")
KEYS = ("mean", "C", "p_sigma", "p_c", "B", "D", "weights", "scalars")


def _fitness(x):
    return (-((x - 0.3) ** 2).sum(-1) + 0.1 * np.sin(5 * x).sum(-1)).astype(np.float32)


def _bits(a, b):
    return np.array_equal(np.asarray(a, dtype=np.float32).view(np.uint32), np.asarray(b, dtype=np.float32).view(np.uint32))


@pytest.mark.skipif(not have_ref(), reason="oracle/_ref/libcmaes_ref.so not built")
@pytest.mark.parametrize("n,lam", [(24, 20), (37, 9), (673, 12)])
def test_restatement_equals_the_reference_objects_bit_for_bit(n, lam):
    a, r = CmaEsOracle(n, lam), CmaEsReference(n, lam)
    sa, sr = a.state(), r.state()
    assert all(_bits(sa[k], sr[k]) for k in KEYS)
    assert (sr["dtypes"] == 6).all()  # the state stays float32; only the arithmetic inside tell is promoted
    for g in range(5 if n < 100 else 2):
        torch.manual_seed(50 + g)
        xa = a.sample()
        torch.manual_seed(50 + g)
        xr = r.sample()
        assert torch.equal(xa, xr), f"generation {g}: samples differ"
        f = _fitness(xr.numpy())
        a.tell(xa, f)
        r.tell(xr, f)
        sa, sr = a.state(), r.state()
        for k in KEYS:
            assert _bits(sa[k], sr[k]), f"generation {g}: {k}"


def test_restatement_equals_golden_vectors():
    z = np.load(GOLDEN)
    n, lam = z["g0_x"].shape[1], z["g0_x"].shape[0]
    a = CmaEsOracle(n, lam)
    for k in KEYS:
        assert _bits(a.state()[k], z[f"init_{k}"]), k
    g = 0
    while f"g{g}_x" in z:
        torch.manual_seed(1000 + g)
        x = a.sample()
        assert _bits(x.numpy(), z[f"g{g}_x"]), f"generation {g}: samples"
        a.tell(x, z[f"g{g}_fit"])
        for k in KEYS:
            assert _bits(a.state()[k], z[f"g{g}_{k}"]), f"generation {g}: {k}"
        g += 1
    assert g >= 8


def test_controller_restatement_and_population_controller():
    z = np.load(GOLDEN)
    for rays in (5, 32, 128):
        flat, obs, want = z[f"ctrl{rays}_flat"], z[f"ctrl{rays}_obs"], z[f"ctrl{rays}_out"]
        got = np.stack([controller_forward(flat[i], obs[i], rays) for i in range(len(flat))])
        assert _bits(got, want), f"{rays} rays: restatement vs reference Controller"
        if have_ref():
            assert _bits(reference_controller_forward(flat, obs, rays), want)
        pc = PopulationController(rays)
        assert pc.num_params == flat.shape[1]
        batched = pc.forward(torch.from_numpy(flat), torch.from_numpy(obs)).numpy()
        # bmm sums in another order than Linear: 1e-6 absolute on tanh outputs in [-1, 1]
        assert np.allclose(batched, want, rtol=0, atol=1e-6), rays


def test_product_solver_follows_the_restatement():
    """same z, same fitness -> the batched solver's state tracks the restatement's to float32 rounding: the only
    differences are where the binary64 sums are narrowed (once vs after every candidate) and GEMM summation order.
    Tolerances: mean 1e-6 abs, C 2e-6 abs (entries are O(1)), sigma 1e-6 rel after each of 6 generations."""
    n, lam = 24, 20
    a, b = CmaEs(n, lam, device="cpu"), CmaEsOracle(n, lam)
    assert np.allclose(a.weights.numpy(), b.weights.numpy(), rtol=1e-6, atol=0)
    for k, v in (("mu_eff", 1), ("c_sigma", 2), ("d_sigma", 3), ("c_c", 4), ("c_1", 5), ("c_mu", 6), ("chi_n", 7)):
        assert getattr(a, k) == pytest.approx(float(b.state()["scalars"][v]), rel=1e-6), k
    rng = np.random.default_rng(0)
    for gen in range(6):
        # feed both the SAME candidates (the restatement's): eigenvectors of a near-identity C are ill-conditioned, so
        # samples are compared through the covariance they realise, not vector by vector
        z = torch.from_numpy(rng.standard_normal((lam, n)).astype(np.float32))
        xb = b.sample(z)
        a.sample(z)
        assert np.allclose(((a.B * a.D**2) @ a.B.t()).numpy(), ((b.B * b.D**2) @ b.B.t()).numpy(), rtol=1e-4, atol=1e-5)
        fit = _fitness(xb.numpy())
        a.tell(xb, torch.from_numpy(fit))
        b.tell(xb, fit)
        assert np.allclose(a.mean.numpy(), b.mean.numpy(), rtol=0, atol=1e-6), gen
        assert np.allclose(a.C.numpy(), b.C.numpy(), rtol=0, atol=2e-6), gen
        assert np.allclose(a.p_sigma.numpy(), b.p_sigma.numpy(), rtol=0, atol=2e-5), gen
        assert np.allclose(a.p_c.numpy(), b.p_c.numpy(), rtol=0, atol=1e-5), gen
        assert a.sigma == pytest.approx(b.sigma, rel=1e-6), gen


def test_ranks_draw_distinct_candidates():
    """round-1 advisor finding: every rank seeded its generator identically, so the 'population' was world copies of
    lambda / world candidates.  With `seed` the solver folds the rank in."""
    a = CmaEs(6, 8, device="cpu", seed=1)
    b = CmaEs(6, 8, device="cpu", seed=1)
    b.rank = 1
    b.gen = torch.Generator(device="cpu").manual_seed(1 * 1_000_003 + 1)  # what rank 1 builds
    assert not torch.equal(a.sample(), b.sample())
    with pytest.raises(ValueError):
        CmaEs(6, 8, device="cpu", seed=1, generator=torch.Generator())
