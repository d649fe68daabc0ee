"""CPU tests (no GPU needed): the C-ABI library loads and exports every symbol
include/ehmc.h declares; the host-side mirror of the reference's classes behaves like
the reference where no compute is involved; compute calls fail loudly without a GPU."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import physicsbasedbayesianinference_b200 as E
from physicsbasedbayesianinference_b200 import _lib
from physicsbasedbayesianinference_b200.build import cuda_tool

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "ehmc.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ehmc_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_all_exported():
    lib = _lib.load()
    declared = _declared_symbols()
    assert declared, "no declarations parsed from include/ehmc.h"
    assert sorted(_lib.SYMBOLS) == declared
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in ehmc.h but not exported by _ehmc.so"
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r"\bT (ehmc_[a-z0-9_]+)", out))
    assert exported == set(declared), exported ^ set(declared)


def test_version_and_struct_layout():
    assert _lib.load().ehmc_version() == 110
    # struct ehmc_hmc_args: 4 x 32-bit, 4 doubles, 3 x u64, 1 pointer; struct ehmc_dynamic: 2 doubles, 3 x u64
    assert ctypes.sizeof(_lib.HmcArgs) == 16 + 32 + 24 + 8
    assert ctypes.sizeof(_lib.Dynamic) == 40
    a = _lib.make_args(0.1, 0.1**2, int(1.0 / 0.1), 1.380649e-23, 300.0, seed=(1 << 40) + 5, iteration=7)
    assert a.struct_size == ctypes.sizeof(_lib.HmcArgs) and a.numSteps == 10 and a.seed == (1 << 40) + 5


def test_library_contains_sm100a_sass_only():
    out = subprocess.run([cuda_tool("cuobjdump"), "-lelf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    assert not re.search(r"sm_(?!100a)\d+", out)


def test_no_cpu_fallback_without_gpu():
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(_lib.EhmcError, match="no CPU fallback"):
        _lib.Context.get()
    ens = E.Ensemble(2, 4)
    integ = E.Leapfrog(ens, 0.1, 1.0, E.HarmonicPotential([1.0, 1.0]))
    with pytest.raises(_lib.EhmcError):
        integ.integrate()
    with pytest.raises(_lib.EhmcError):
        E.harmonicPotentialND(ens.q, np.array([2.0, 3.0]))


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "physicsbasedbayesianinference_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+\.*oracle\b", text, flags=re.M), f
                assert not re.search(r"(import_module|__import__|CDLL)\([^)]*oracle", text), f


# ---- Ensemble (src/ensemble.py, src/tests/test_ensemble.py) ---------------------------------
def test_ensemble_init_KA2():
    ens = E.Ensemble(4, 100)
    q1, p1, m1, w1 = ens.particle(10)
    assert np.all(q1 == 0) and np.all(p1 == 0) and m1 == 1.0 and w1 == 0.0
    assert ens.q.shape == (4, 100) and ens.q.dtype == np.float64 and ens.q.flags.c_contiguous
    with pytest.raises(IndexError):
        ens.particle(101)
    with pytest.raises(IndexError):
        ens.particle(-1)
    q, p, m, w = ens  # unpacking works (the reference's __iter__ raises AttributeError)
    assert q is ens.q and w is ens.weights


def test_ensemble_host_rng_is_the_reference_stream():
    """setPosition / setMomentum consume NumPy's global MT19937 like scipy's norm.rvs in
    src/ensemble.py:72-74,88-91 (SURVEY rows B, C): bit-equal to standard_normal * scale."""
    kB = 1.380649e-23
    np.random.seed(5)
    ens = E.Ensemble(3, 7)
    ens.mass = np.linspace(1, 2, 7)
    q = ens.setPosition(2.5)
    p = ens.setMomentum(300.0)
    assert q is ens.q and p is ens.p
    np.random.seed(5)
    assert np.array_equal(q, np.random.standard_normal((3, 7)) * 2.5)
    assert np.array_equal(p, np.random.standard_normal((3, 7)) * np.sqrt(ens.mass * kB * 300.0))


# ---- Integrator / HMC construction (no compute) ---------------------------------------------
@pytest.mark.parametrize("ft,h,n", [(0.3, 0.1, 2), (1.0, 0.05, 20), (2.5, 0.05, 50), (0.5, 0.05, 10)])
def test_num_steps_float_floor(ft, h, n):
    """src/integrator.py:51: int(finalTime / stepSize), e.g. int(0.3/0.1) == 2."""
    ens = E.Ensemble(2, 4)
    assert E.Leapfrog(ens, h, ft, E.HarmonicPotential([1.0, 1.0])).numSteps == n == int(ft / h)


def test_integrator_aliases_ensemble_arrays():
    ens = E.Ensemble(2, 4)
    ens.p[:] = 3.0
    ens.mass = np.array([1.0, 2.0, 3.0, 6.0])
    integ = E.StormerVerlet(ens, 0.1, 1.0, E.HarmonicPotential([1.0, 1.0]).gradient)
    assert integ.q is ens.q and integ.p is ens.p and integ.mass is ens.mass
    assert np.array_equal(integ.v, ens.p / ens.mass)
    assert integ.numParticles == 4 and integ.stepSize == 0.1 and integ.finalTime == 1.0


def test_hmc_constructor_errors_and_method_selection():
    ens = E.Ensemble(2, 4)
    pot = E.HarmonicPotential([1.0, 1.0])
    assert isinstance(E.HMC(ens, 1.0, 0.1, None, potential=pot).integrator, E.Leapfrog)
    assert isinstance(E.HMC(ens, 1.0, 0.1, None, gradient=pot.gradient, method="Stormer-Verlet").integrator,
                      E.StormerVerlet)
    assert isinstance(E.HMC(ens, 1.0, 0.1, E.GaussianDensity([0, 0], np.eye(2))).integrator, E.Leapfrog)
    with pytest.raises(ValueError, match="Invalid integration method selected."):
        E.HMC(ens, 1.0, 0.1, None, potential=pot, method="RK4")
    with pytest.raises(TypeError, match="no CPU fallback"):
        E.HMC(ens, 1.0, 0.1, lambda q: np.exp(-0.5 * q @ q))
    with pytest.raises(NotImplementedError):
        E.Integrator(ens, 0.1, 1.0, pot).integrate()


def test_nbody_mode_constructor_prints_like_reference(capsys):
    ens = E.Ensemble(3, 3)
    integ = E.Leapfrog(ens, 600, 3600, None)
    assert "Gradient=None - performing nBody simulation." in capsys.readouterr().out
    assert integ.nBodyMode and integ.numSteps == 6


def test_flat_module_shims(tmp_path):
    code = ("import sys; sys.path.insert(0, %r); from ensemble import Ensemble; from integrator import Leapfrog, "
            "StormerVerlet; from HMC import HMC; from potential import harmonicPotentialND, noPotential; "
            "print(Ensemble(2, 3).q.shape, noPotential(0))") % os.path.join(
                ROOT, "physicsbasedbayesianinference_b200", "flat")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=tmp_path)
    assert out.returncode == 0, out.stderr
    assert "(2, 3) 0" in out.stdout


# ---- section 8f rows: input files, checkpoints, model adapter (host logic) -------------------
def test_read_nbody_input_reference_files(tmp_path):
    """ReadInput format of samples/NBody/MiscFunctions.py:8-43 (copy of pl3.txt's numbers)."""
    from physicsbasedbayesianinference_b200 import io

    txt = (" 3  220.0       0.1     \n0.99990\n0.00001\n0.00009\n0.0      0.0       0.0\n1.0      0.0       0.0\n"
           "-2.25    0.0       0.0\n0.0      0.0       0.0     \n0.0     -1.0       0.0\n0.0      0.6666666    0.0\n")
    f = tmp_path / "pl3.txt"
    f.write_text(txt)
    N, tmax, dt, M, PS = io.readNBodyInput(str(f))
    assert (N, tmax, dt) == (3, 220.0, 0.1)
    assert np.allclose(M, [0.9999, 0.00001, 0.00009])
    assert np.allclose(PS[:, 0, 0], [0.0, 1.0, -2.25]) and np.allclose(PS[:, 1, 1], [0.0, -1.0, 0.6666666])
    q, p = io.nbodyInputToEnsembleColumn(M, PS)
    assert q.shape == (9,) and np.allclose(q[:3], [0.0, 1.0, -2.25]) and np.allclose(p[3:6], M * PS[:, 1, 1])
    f.write_text(" 3 1.0 0.1\n1\n2\n")
    with pytest.raises(ValueError):
        io.readNBodyInput(str(f))


def test_checkpoint_roundtrip_host(tmp_path):
    from physicsbasedbayesianinference_b200 import io

    ens = E.Ensemble(2, 5)
    ens.q[:] = np.arange(10).reshape(2, 5)
    ens.mass = np.linspace(1, 2, 5)
    hmc = E.HMC(ens, 1.0, 0.1, None, potential=E.HarmonicPotential([1.0, 2.0]), rng="philox", seed=77)
    hmc.iteration = 41
    io.saveCheckpoint(str(tmp_path / "ck"), hmc)
    ens2 = E.Ensemble(2, 5)
    hmc2 = E.HMC(ens2, 1.0, 0.25, None, potential=E.HarmonicPotential([1.0, 2.0]), rng="philox", seed=1)
    io.loadCheckpoint(str(tmp_path / "ck"), hmc2)
    assert np.array_equal(ens2.q, ens.q) and np.array_equal(ens2.mass, ens.mass)
    assert (hmc2.seed, hmc2.iteration, hmc2.stepSize, hmc2.integrator.numSteps) == (77, 41, 0.1, 10)


def test_model_spec_adapter():
    from physicsbasedbayesianinference_b200 import numpyro_adapter as A

    p = A.potentialFromSpec(dict(family="normal_iid", scale=[1.0, 0.5]))
    assert isinstance(p, E.HarmonicPotential) and np.allclose(p.springConsts, [1.0, 4.0])
    p = A.potentialFromSpec(dict(family="mvn", mean=[5, 5], cov=[[4, -3], [-3, 4]]))
    assert isinstance(p, E.GaussianPotential) and np.allclose(p.precision @ [[4, -3], [-3, 4]], np.eye(2))
    assert isinstance(A.potentialFromSpec(dict(family="funnel", numDimensions=10)), E.FunnelPotential)
    X = np.ones((4, 3))
    assert A.potentialFromSpec(dict(family="logistic_regression", X=X, y=np.ones(4))).numDimensions == 3
    # the reference's own NumPyro sample model (CoinToss.data.json: c1, c2)
    p = A.potentialFromSpec(dict(family="coin_toss", observations=[[1, 0] * 10, [1] * 15 + [0] * 5]))
    assert isinstance(p, E.CoinTossPotential) and list(p.successes) == [10, 15] and list(p.trials) == [20, 20]
    with pytest.raises(NotImplementedError):
        A.potentialFromSpec(dict(family="eight_schools"))
    with pytest.raises((ImportError, NotImplementedError)):
        A.potentialFromNumpyroModel(lambda: None)


def test_logistic_recognition_from_logits():
    """The Bernoulli-logit recogniser of the NumPyro adapter (the part that needs no NumPyro): X is recovered from
    the logits of the observed site, models with an intercept or a non-linear predictor are refused."""
    from physicsbasedbayesianinference_b200 import numpyro_adapter as A

    rng = np.random.RandomState(5)
    X = rng.standard_normal((50, 4))
    y = (rng.uniform(size=50) < 0.5).astype(np.float64)
    spec = A.logisticSpecFromLinearLogits(lambda th: X @ th, 4, y, 2.0)
    assert spec["family"] == "logistic_regression" and spec["priorScale"] == 2.0
    np.testing.assert_allclose(spec["X"], X, rtol=0, atol=1e-15)
    pot = A.potentialFromSpec(spec)
    assert pot.numDimensions == 4
    with pytest.raises(NotImplementedError):
        A.logisticSpecFromLinearLogits(lambda th: X @ th + 0.3, 4, y, 1.0)  # intercept
    with pytest.raises(NotImplementedError):
        A.logisticSpecFromLinearLogits(lambda th: np.tanh(X @ th), 4, y, 1.0)  # not linear
    with pytest.raises(NotImplementedError):
        A.logisticSpecFromLinearLogits(lambda th: X @ th, 4, y + 0.5, 1.0)  # not 0/1 observations


def test_checkpoint_round_trip_of_driver_state_on_host(tmp_path):
    """saveCheckpoint / loadCheckpoint carry everything the next call depends on: positions, masses, Philox (seed,
    iteration), step size, the trajectory length actually in use (numSteps and the simulTime that drifted with it),
    the flags and the mass scales (no GPU needed: nothing is launched)."""
    ens = E.Ensemble(3, 16)
    ens.q[:] = np.arange(48.0).reshape(3, 16)
    ens.mass[:] = 2.0
    hmc = E.HMC(ens, 1.0, 0.1, None, potential=E.HarmonicPotential(np.ones(3)), bugCompat=False, rejectNonFinite=True)
    hmc.iteration, hmc.stepSize = 77, 0.25
    hmc.integrator.stepSize, hmc.integrator.numSteps = 0.25, 10
    hmc.simulTime = hmc.integrator.finalTime = 2.5
    hmc.massScale = np.array([1.0, 2.0, 4.0])
    E.io.saveCheckpoint(str(tmp_path / "ck"), hmc)
    ens2 = E.Ensemble(3, 16)
    hmc2 = E.HMC(ens2, 1.0, 0.1, None, potential=E.HarmonicPotential(np.ones(3)))
    E.io.loadCheckpoint(str(tmp_path / "ck"), hmc2)
    assert np.array_equal(ens2.q, ens.q) and np.array_equal(ens2.mass, ens.mass)
    assert hmc2.integrator.q is ens2.q and hmc2.iteration == 77 and hmc2.seed == hmc.seed
    assert hmc2.stepSize == 0.25 and hmc2.integrator.stepSize == 0.25
    assert hmc2.integrator.numSteps == 10 and hmc2.simulTime == 2.5 and hmc2.integrator.finalTime == 2.5
    assert hmc2.bugCompat is False and hmc2.rejectNonFinite is True
    np.testing.assert_array_equal(hmc2.massScale, [1.0, 2.0, 4.0])
    hmc.rejectNonFinite, hmc.massScale = None, None
    E.io.saveCheckpoint(str(tmp_path / "ck2"), hmc)
    E.io.loadCheckpoint(str(tmp_path / "ck2"), hmc2)
    assert hmc2.rejectNonFinite is None and hmc2.massScale is None
    with pytest.raises(ValueError):
        E.io.loadCheckpoint(str(tmp_path / "ck2"), E.HMC(E.Ensemble(3, 8), 1.0, 0.1, None, potential=E.HarmonicPotential(np.ones(3))))


def test_run_argument_validation_without_a_gpu():
    """HMC.run refuses inconsistent requests before anything is launched."""
    ens = E.Ensemble(2, 8)
    hmc = E.HMC(ens, 1.0, 0.1, None, potential=E.HarmonicPotential(np.ones(2)))
    with pytest.raises(ValueError):
        hmc.run(1, 1.0, adaptLag=5)
    with pytest.raises(ValueError):
        hmc.run(1, 1.0, adaptMass=True)  # needs adapt=True
    with pytest.raises(ValueError):
        hmc.run(1, 1.0, adapt=True, deviceAdapt=True, adaptLag=2)
    assert hmc._inRun is False  # the guard of run() is released on every exit path
