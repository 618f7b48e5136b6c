"""CPU-side tests: the C-ABI library loads and exports every symbol include/smcb.h
declares, the host logic that maps Feynman-Kac objects onto fused kernels, the Philox
restatement used by the GPU tests, and the no-CPU-fallback rule.  No compute calls."""
import ctypes
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import philox_ref  # noqa: E402


@pytest.fixture(scope="module")
def lib():
    from particles_b200 import _lib, build
    build.build()
    return _lib.load()


def header_symbols():
    txt = open(os.path.join(ROOT, "include", "smcb.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(smcb_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol(lib):
    from particles_b200 import _lib
    syms = header_symbols()
    assert len(syms) >= 25
    raw = ctypes.CDLL(_lib.SO_PATH)
    for s in syms:
        assert hasattr(raw, s), f"{s} declared in include/smcb.h but not exported"
    assert set(_lib.PROTOTYPES) == set(syms)          # the ctypes layer binds exactly the header
    assert lib.smcb_version() == 100
    assert lib.smcb_resample_scratch_doubles(1000, 500) >= 1000 + 500


def test_built_for_sm_100a_only():
    from particles_b200 import _lib, build
    nvcc = shutil.which(build._nvcc())
    assert nvcc, f"{build._nvcc()} not found: the CUDA toolkit that built the library is needed to inspect it"
    cuobjdump = os.path.join(os.path.dirname(nvcc), "cuobjdump")   # from the toolkit that built the library
    out = subprocess.run([cuobjdump, "-lelf", _lib.SO_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_filter_desc_layout_matches_header():
    """ctypes mirror of smcb_filter_desc: every field at the same offset as in the C struct."""
    from particles_b200 import _lib
    D = _lib.FilterDesc
    names = [f[0] for f in D._fields_]
    probes = ", ".join(f"offsetof(smcb_filter_desc, {n})" for n in names)
    fmt = " ".join(["%zu"] * (len(names) + 1))
    src = f'''
    #include <stdio.h>
    #include <stddef.h>
    #include "smcb.h"
    int main(void) {{ printf("{fmt}\\n", sizeof(smcb_filter_desc), {probes}); return 0; }}
    '''
    exe = os.path.join(ROOT, "oracle", "_build", "layout_probe")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    subprocess.run(["gcc", "-x", "c", "-", "-I", os.path.join(ROOT, "include"), "-o", exe],
                   input=src, text=True, check=True)
    vals = [int(v) for v in subprocess.run([exe], capture_output=True, text=True).stdout.split()]
    assert vals[0] == ctypes.sizeof(D)
    assert dict(zip(names, vals[1:])) == {n: getattr(D, n).offset for n in names}


def test_philox_known_answers():
    """Random123 known-answer vectors for philox4x32-10."""
    def k(c, key):
        return [int(v) for v in philox_ref.philox4x32_10(*[np.uint32(x) for x in c], key[0], key[1])]
    assert k([0, 0, 0, 0], [0, 0]) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert k([0xffffffff] * 4, [0xffffffff] * 2) == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert k([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0]) == \
        [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]
    u = philox_ref.uniforms(10001, 3, 42)
    assert u.min() >= 0 and u.max() < 1 and abs(u.mean() - 0.5) < 0.02


def test_fused_spec_recognition():
    from particles_b200 import _lib, kalman, state_space_models as ssm
    y = [np.array([0.1 * i]) for i in range(7)]
    s = ssm.fused_spec(ssm.Bootstrap(ssm=ssm.StochVol(), data=y))
    assert s["model"] == _lib.MODEL_STOCHVOL and s["fk"] == _lib.FK_BOOTSTRAP
    assert s["data"].shape == (7, 1) and s["params"][4] == (1.0 - 0.9702) * -1.02
    assert ssm.fused_spec(ssm.AuxiliaryPF(ssm=ssm.StochVol(), data=y))["fk"] == _lib.FK_APF
    assert ssm.fused_spec(ssm.GuidedPF(ssm=kalman.LinearGauss(), data=y))["model"] == _lib.MODEL_LINGAUSS
    g = ssm.fused_spec(ssm.Bootstrap(ssm=ssm.Gordon_etal(), data=y))
    assert np.array_equal(g["step_consts"], [8.0 * np.cos(1.2 * (t - 1)) for t in range(7)])
    # no proposal -> not fused as guided; user subclasses are never taken for stock models
    assert ssm.fused_spec(ssm.GuidedPF(ssm=ssm.Gordon_etal(), data=y)) is None

    class MySV(ssm.StochVol):
        def PY(self, t, xp, x):
            return None
    MySV.__module__ = "user_code"
    assert ssm.fused_spec(ssm.Bootstrap(ssm=MySV(), data=y)) is None

    class MyFK(ssm.Bootstrap):
        pass
    assert ssm.fused_spec(MyFK(ssm=ssm.StochVol(), data=y)) is None
    with pytest.raises(ValueError):
        ssm.fused_spec(ssm.Bootstrap(ssm=ssm.StochVol(), data=[np.zeros(2)] * 3))


def _reference_model(g, name):
    """A model object as the reference builds it: class name, module and instance attributes recorded from the
    reference in tests/golden/golden_dropin.npz (make_golden_dropin.py)."""
    cls = type(name, (), {"__module__": str(g[f"model/{name}/module"])})
    obj = cls()
    prefix = f"model/{name}/attr/"
    for key in g.files:
        if key.startswith(prefix):
            v = g[key]
            setattr(obj, key[len(prefix):], v.item() if v.ndim == 0 else v)
    return obj


def _reference_fk(g, name, ssm, data):
    """A Feynman-Kac object of the reference's class ``name``: same class names along the method resolution order."""
    base = None
    for nm in reversed([str(s) for s in g[f"fk/{name}/mro"]]):
        base = type(nm, () if base is None else (base,), {})
    fk = base()
    fk.ssm, fk.data, fk.T = ssm, data, len(data)
    return fk


def test_reference_objects_are_recognised():
    """Drop-in: a Feynman-Kac object built from the REFERENCE's own classes maps onto the
    same fused kernel constants as ours."""
    from particles_b200 import kalman, state_space_models as ssm
    g = np.load(os.path.join(ROOT, "tests", "golden", "golden_dropin.npz"))
    y = [np.array([0.3 * i]) for i in range(5)]
    for name, ours in [("StochVol", ssm.StochVol(mu=-0.5)), ("LinearGauss", kalman.LinearGauss(rho=0.7)),
                       ("Gordon_etal", ssm.Gordon_etal()), ("ThetaLogistic", ssm.ThetaLogistic())]:
        a = ssm.fused_spec(_reference_fk(g, "Bootstrap", _reference_model(g, name), y))
        b = ssm.fused_spec(ssm.Bootstrap(ssm=ours, data=y))
        assert a["model"] == b["model"] and a["fk"] == b["fk"] and list(a["params"]) == list(b["params"])
        assert np.array_equal(a["data"], b["data"])
    assert ssm.fused_spec(_reference_fk(g, "AuxiliaryPF", _reference_model(g, "StochVol"), y))["fk"] == 2


def test_no_cpu_fallback():
    """Without a CUDA device the product raises; it never computes on the host."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import particles_b200 as pb
    from particles_b200 import _lib, resampling as rs, state_space_models as ssm
    with pytest.raises(_lib.SmcbError):
        pb.SMC(fk=ssm.Bootstrap(ssm=ssm.StochVol(), data=[np.zeros(1)] * 3), N=10)
    with pytest.raises(_lib.SmcbError):
        rs.systematic(np.full(4, 0.25))
    with pytest.raises(_lib.SmcbError):
        rs.Weights(lw=np.zeros(3))


def test_product_never_imports_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "particles_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in txt and "from oracle" not in txt, f


def test_collectors_surface():
    from particles_b200 import collectors
    s = collectors.Summaries([collectors.Moments()])
    assert hasattr(s, "ESSs") and hasattr(s, "logLts") and hasattr(s, "rs_flags") and hasattr(s, "moments")
    assert not s.only_defaults and collectors.Summaries(None).only_defaults
    with pytest.raises(ValueError):
        collectors.Moments(bogus=1)
