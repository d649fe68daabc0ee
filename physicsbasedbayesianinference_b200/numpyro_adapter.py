"""NumPyro-model -> potential-family adapter (SURVEY.md section 8f row 2).

The reference intends potentials built from a NumPyro model through
``-numpyro.infer.util.log_density(model, args, kwargs, params)[0]`` and ``jax.grad`` of it
(samples/NumpyroExamples/CoinToss/CoinTossExample.py:75-107).  A fused CUDA trajectory kernel
cannot trace an arbitrary model, so the adapter RECOGNISES the model families the engine has
kernels for and raises for everything else.  NumPyro / JAX are optional imports (absent in the
build image); recognition works on a declarative spec so it is testable without them.
"""
from __future__ import annotations

import numpy as np

from .potential import (CoinTossPotential, FunnelPotential, GaussianPotential, HarmonicPotential,
                        HierarchicalNormalPotential, LogisticPotential)


def potentialFromSpec(spec):
    """spec: dict(family=..., **parameters) -> potential descriptor.

    families: "normal_iid" (scale per dim), "mvn" (mean, cov | precision),
    "funnel" (numDimensions, sigmaV), "coin_toss" (observations | successes, trials),
    "logistic_regression" (X, y, priorScale),
    "hierarchical_normal" (y, sigma, muLoc, muScale, tauScale, centered)."""
    fam = spec.get("family")
    if fam == "normal_iid":
        scale = np.atleast_1d(np.asarray(spec["scale"], dtype=np.float64))
        return HarmonicPotential(1.0 / scale**2)
    if fam == "mvn":
        if "precision" in spec:
            return GaussianPotential(precision=spec["precision"], mean=spec.get("mean"))
        return GaussianPotential(cov=spec["cov"], mean=spec.get("mean"))
    if fam == "funnel":
        return FunnelPotential(int(spec["numDimensions"]), float(spec.get("sigmaV", 3.0)))
    if fam == "coin_toss":  # Uniform(0, 1) priors, Bernoulli observations (CoinToss.py:21-25)
        if "observations" in spec:
            return CoinTossPotential.fromObservations(*spec["observations"])
        return CoinTossPotential(spec["successes"], spec["trials"])
    if fam == "logistic_regression":
        return LogisticPotential(spec["X"], spec["y"], float(spec.get("priorScale", 1.0)),
                                 precision=spec.get("precision", "fp32"))
    if fam == "hierarchical_normal":  # eight schools: HierarchicalNormalPotential.eightSchools()
        return HierarchicalNormalPotential(spec["y"], spec["sigma"], float(spec.get("muLoc", 0.0)),
                                           float(spec.get("muScale", 5.0)), float(spec.get("tauScale", 5.0)),
                                           spec.get("centered", False))
    raise NotImplementedError(
        f"model family {fam!r} has no fused CUDA kernel; supported: normal_iid, mvn, funnel, coin_toss, "
        "logistic_regression, hierarchical_normal")


def logisticSpecFromLinearLogits(logits_of, numDimensions, y, priorScale, rtol=1e-6):
    """Recognises ``obs ~ Bernoulli(logits = X @ theta)`` from the logits alone and returns the
    ``logistic_regression`` spec (the design matrix is not visible in a model trace, only the logits are).

    logits_of(theta) -> logits (N,) of the observed site with the latent vector fixed to theta.  X is recovered by
    probing the unit vectors, column k = logits_of(e_k) - logits_of(0); the model is accepted only if it has no
    intercept (logits_of(0) == 0: the family has none) and is linear (checked on a random theta).  Raises
    NotImplementedError otherwise."""
    D = int(numDimensions)
    base = np.asarray(logits_of(np.zeros(D)), dtype=np.float64).reshape(-1)
    if not np.allclose(base, 0.0, atol=1e-12):
        raise NotImplementedError("Bernoulli-logit model with an intercept / offset: the logistic family is X @ theta only")
    X = np.empty((base.shape[0], D))
    for k in range(D):
        e = np.zeros(D)
        e[k] = 1.0
        X[:, k] = np.asarray(logits_of(e), dtype=np.float64).reshape(-1)
    th = np.random.RandomState(0).standard_normal(D)
    got = np.asarray(logits_of(th), dtype=np.float64).reshape(-1)
    want = X @ th
    if not np.allclose(got, want, rtol=rtol, atol=rtol * max(1.0, float(np.max(np.abs(want))))):
        raise NotImplementedError("the logits of the observed Bernoulli site are not linear in the latent vector")
    y = np.asarray(y, dtype=np.float64).reshape(-1)
    if y.shape[0] != X.shape[0] or not np.all((y == 0) | (y == 1)):
        raise NotImplementedError("observations must be one 0/1 value per row of the design matrix")
    return dict(family="logistic_regression", X=X, y=y, priorScale=float(priorScale))


def potentialFromNumpyroModel(model, model_args=(), model_kwargs=None):
    """Traces a NumPyro model once and maps it to a family (needs numpyro + jax).  Recognised:
    a single MultivariateNormal / Normal latent site without observations, and a Bernoulli-logit
    likelihood ``obs ~ Bernoulli(logits = X @ theta)`` with a Normal(0, s) prior on theta
    (logisticSpecFromLinearLogits), and the coin-toss sample of the reference.

    NumPyro and JAX are absent from the build image, so this function itself has never run there: the
    recognisers it delegates to (potentialFromSpec, logisticSpecFromLinearLogits) are what the tests cover."""
    try:
        import numpyro  # noqa: F401
        from numpyro import handlers
        import numpyro.distributions as dist
        import jax
    except ImportError as e:  # pragma: no cover - numpyro is not in the build image
        raise ImportError("potentialFromNumpyroModel needs numpyro and jax; use potentialFromSpec instead") from e
    tr = handlers.trace(handlers.seed(model, jax.random.PRNGKey(0))).get_trace(*model_args, **(model_kwargs or {}))
    latent = [s for s in tr.values() if s["type"] == "sample" and not s["is_observed"]]
    observed = [s for s in tr.values() if s["type"] == "sample" and s["is_observed"]]
    if latent and len(latent) == len(observed) and all(
            isinstance(s["fn"], dist.Uniform) and float(s["fn"].low) == 0.0 and float(s["fn"].high) == 1.0 for s in latent) and all(
            isinstance(getattr(s["fn"], "base_dist", s["fn"]), (dist.BernoulliProbs,)) for s in observed):
        # the coin-toss sample: site k observes Bernoulli(latent k)
        return potentialFromSpec(dict(family="coin_toss", observations=[np.asarray(s["value"]) for s in observed]))
    if len(latent) == 1 and len(observed) == 1:
        # Bayesian logistic regression: theta ~ Normal(0, s) iid, obs ~ Bernoulli(logits = X @ theta)
        prior = getattr(latent[0]["fn"], "base_dist", latent[0]["fn"])
        like = getattr(observed[0]["fn"], "base_dist", observed[0]["fn"])
        scale = np.unique(np.asarray(getattr(prior, "scale", np.nan), dtype=np.float64))
        if (isinstance(prior, dist.Normal) and np.allclose(np.asarray(prior.loc), 0.0) and scale.size == 1
                and isinstance(like, dist.BernoulliLogits) and np.ndim(latent[0]["value"]) == 1):
            name, obs_name = latent[0]["name"], observed[0]["name"]

            def logits_of(theta):
                t = handlers.trace(handlers.substitute(handlers.seed(model, jax.random.PRNGKey(0)), {name: jax.numpy.asarray(theta)}))
                site = t.get_trace(*model_args, **(model_kwargs or {}))[obs_name]
                return np.asarray(getattr(site["fn"], "base_dist", site["fn"]).logits)

            return potentialFromSpec(logisticSpecFromLinearLogits(logits_of, latent[0]["value"].shape[0],
                                                                  np.asarray(observed[0]["value"]), float(scale[0])))
    if len(latent) == 1 and not observed:
        d = latent[0]["fn"]
        if isinstance(d, dist.MultivariateNormal):
            return potentialFromSpec(dict(family="mvn", mean=np.asarray(d.mean), cov=np.asarray(d.covariance_matrix)))
        base = getattr(d, "base_dist", d)
        if isinstance(base, dist.Normal) and np.allclose(np.asarray(base.loc), 0.0):
            return potentialFromSpec(dict(family="normal_iid", scale=np.broadcast_to(np.asarray(base.scale), latent[0]["value"].shape)))
    raise NotImplementedError("this NumPyro model does not match a family with a fused CUDA kernel; "
                              "describe it with potentialFromSpec(dict(family=...)) if it is one of them")
