"""The literal drop-in: ``particles_b200.install()`` rebinds ``particles.SMC`` and the REFERENCE's own model /
Feynman-Kac objects run on the fused kernels.  On a box that has the live reference (oracle/_ref, copied by
oracle/make_ref.sh in the build container; never part of the repository) the real classes are used; otherwise a
stand-in package with the same module and class names and the same attributes is put into sys.modules."""
import os
import sys
import types

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

from oracle import smc_numpy as orc  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref")


def _stand_in():
    """particles / particles.core / particles.state_space_models with the reference's class names."""
    pkg, core, ssm = types.ModuleType("particles"), types.ModuleType("particles.core"), \
        types.ModuleType("particles.state_space_models")

    class SMC:                                    # what install() replaces
        def __init__(self, *a, **k):
            raise RuntimeError("the stand-in reference has no engine")

    class StochVol:
        def __init__(self, mu=-1.02, rho=0.9702, sigma=0.178):
            self.mu, self.rho, self.sigma = mu, rho, sigma

    class Bootstrap:
        def __init__(self, ssm=None, data=None):
            self.ssm, self.data = ssm, data

        @property
        def T(self):
            return len(self.data)

        def done(self, smc):
            return smc.t >= self.T

    for cls, mod in ((SMC, core), (StochVol, ssm), (Bootstrap, ssm)):
        cls.__module__ = mod.__name__
        setattr(mod, cls.__name__, cls)
    pkg.core, pkg.state_space_models, pkg.SMC = core, ssm, SMC
    pkg.__path__ = []
    return {"particles": pkg, "particles.core": core, "particles.state_space_models": ssm}


@pytest.fixture()
def reference(request):
    """(particles module, is_live) with sys.modules restored afterwards."""
    saved = {k: v for k, v in sys.modules.items() if k == "particles" or k.startswith("particles.")}
    for k in saved:
        del sys.modules[k]
    live = os.path.isdir(os.path.join(REF, "particles"))
    if live:
        sys.path.insert(0, REF)
        import particles
    else:
        sys.modules.update(_stand_in())
        import particles
    yield particles, live
    for k in [k for k in sys.modules if k == "particles" or k.startswith("particles.")]:
        del sys.modules[k]
    sys.modules.update(saved)
    if live:
        sys.path.remove(REF)


def test_install_runs_reference_objects_on_the_fused_kernels(reference, golden):
    particles, _ = reference
    import particles_b200 as pb
    import particles.state_space_models as rssm
    N, T = 4096, 40
    y = [np.atleast_1d(v) for v in golden["data/sv_seed1_T1000"][:T]]
    r = np.random.RandomState(3)
    z, u = r.standard_normal((T, N)), r.rand(T, N + 1)
    undo = pb.install()
    try:
        assert particles.SMC is pb.SMC and particles.core.SMC is pb.SMC
        fk = rssm.Bootstrap(ssm=rssm.StochVol(), data=y)          # the REFERENCE's classes
        assert type(fk).__module__ == "particles.state_space_models"
        pf = particles.SMC(fk=fk, N=N, ESSrmin=0.7, noise=(z, u))
        assert pf.fused
        pf.run()
    finally:
        undo()
    assert particles.SMC is not pb.SMC
    ref = orc.SMC(orc.Bootstrap(orc.StochVol(), y), N=N, ESSrmin=0.7,
                  noise=orc.InjectedNoise(z, [row[:1] for row in u])).run()
    assert pf.summaries.rs_flags == ref.rs_flags and sum(ref.rs_flags) > 0
    np.testing.assert_allclose(pf.logLt, ref.logLt, rtol=1e-11)
    assert np.array_equal(pf.X.cpu().numpy(), ref.X) and np.array_equal(pf.A.cpu().numpy(), ref.A)
    # and the reference itself agrees statistically (its own RNG): 3 sigma of its own spread.  Its logLt over 6 seeded
    # runs of the same filter were recorded from the live reference (tests/golden/make_golden_dropin.py)
    g = np.load(os.path.join(ROOT, "tests", "golden", "golden_dropin.npz"))
    assert int(g["stat/N"]) == N and int(g["stat/T"]) == T
    lls = g["stat/logLt"]
    dev = []
    for seed in range(6):
        q = pb.SMC(fk=rssm.Bootstrap(ssm=rssm.StochVol(), data=y), N=N, ESSrmin=0.7, seed=seed)
        q.run()
        dev.append(q.logLt)
    sd = np.std(lls, ddof=1)
    assert abs(np.mean(dev) - np.mean(lls)) < 3 * sd * np.sqrt(2 / 6) + 1e-6, (dev, lls)
