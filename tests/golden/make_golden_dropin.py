"""What the drop-in tests compare against, recorded from the LIVE reference (nchopin/particles):

    PYTHONDONTWRITEBYTECODE=1 PYTHONPATH=<reference checkout> python tests/golden/make_golden_dropin.py

Writes tests/golden/golden_dropin.npz:
* ``model/<class>/module`` and ``model/<class>/attr/<name>``: module and instance attributes of the reference's
  StochVol(mu=-0.5), LinearGauss(rho=0.7), Gordon_etal() and ThetaLogistic() -- everything
  ``particles_b200.state_space_models.fused_spec`` reads from a model object;
* ``fk/<class>/mro``: class names along the method resolution order of the reference's Bootstrap and AuxiliaryPF;
* ``stat/logLt``: logLt of the reference's own particles.SMC, Bootstrap(StochVol()) on the first 40 observations
  of golden_exact.npz ``data/sv_seed1_T1000``, N = 4096, ESSrmin = 0.7, after ``numpy.random.seed(s)`` for each s of
  ``stat/seeds``.
(test_host.py::test_reference_objects_are_recognised, test_gpu_dropin.py)"""
import os

import numpy as np

import particles
from particles import kalman as rk
from particles import state_space_models as rssm

HERE = os.path.dirname(os.path.abspath(__file__))
out = {}
for m in (rssm.StochVol(mu=-0.5), rk.LinearGauss(rho=0.7), rssm.Gordon_etal(), rssm.ThetaLogistic()):
    name = type(m).__name__
    out[f"model/{name}/module"] = np.array(type(m).__module__)
    for k, v in vars(m).items():
        out[f"model/{name}/attr/{k}"] = np.asarray(v)
for cls in (rssm.Bootstrap, rssm.AuxiliaryPF):
    out[f"fk/{cls.__name__}/mro"] = np.array([c.__name__ for c in cls.__mro__ if c is not object])

N, T, seeds = 4096, 40, np.arange(100, 106)
y = [np.atleast_1d(v) for v in np.load(os.path.join(HERE, "golden_exact.npz"))["data/sv_seed1_T1000"][:T]]
lls = []
for s in seeds:
    np.random.seed(s)
    pf = particles.SMC(fk=rssm.Bootstrap(ssm=rssm.StochVol(), data=y), N=N, ESSrmin=0.7)
    pf.run()
    lls.append(pf.logLt)
out.update({"stat/seeds": seeds, "stat/logLt": np.array(lls), "stat/N": np.array(N), "stat/T": np.array(T)})
np.savez_compressed(os.path.join(HERE, "golden_dropin.npz"), **out)
print("wrote golden_dropin.npz:", len(out), "arrays; logLt", np.mean(lls), "+-", np.std(lls, ddof=1))
