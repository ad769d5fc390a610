"""Shared fixtures.  GPU tests carry @pytest.mark.gpu; everything else runs on the CPU-only build box."""
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLD = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def oracle():
    from oracle.oracle_bindings import Oracle

    return Oracle()


@pytest.fixture(scope="session")
def reflib():
    from oracle import ref_bindings

    if not ref_bindings.available():
        pytest.skip("the original SLICER build (oracle/_ref, made by oracle/Makefile from its sources) is absent")
    return ref_bindings.RefLib(ngp=False)


@pytest.fixture(scope="session")
def reflib_ngp():
    from oracle import ref_bindings

    if not ref_bindings.available(ngp=True):
        pytest.skip("the original SLICER build (oracle/_ref, made by oracle/Makefile from its sources) is absent")
    return ref_bindings.RefLib(ngp=True)


@pytest.fixture(scope="session")
def kat():
    with open(os.path.join(GOLD, "kat.json")) as f:
        return json.load(f)


class GoldenCases:
    def __init__(self):
        with open(os.path.join(GOLD, "cases.json")) as f:
            self.meta = json.load(f)
        self.arr = np.load(os.path.join(GOLD, "cases.npz"))

    def names(self):
        return list(self.meta)

    def types(self, name):
        """-> list of dicts ready for Oracle.plane_from_particles / staging."""
        m = self.meta[name]
        out = []
        for t_str, n in sorted(m["npart"].items(), key=lambda kv: int(kv[0])):
            t = int(t_str)
            d = dict(type=t, raw=self.arr[f"{name}/pos{t}"])
            if m["hydro"] and m["massarr"][t] == 0:
                d["masses"] = self.arr[f"{name}/mass{t}"]
                d["cut"] = True
            else:
                d["const_mass"] = m["massarr"][t]
            out.append(d)
        return out

    def plane(self, name):
        m = self.meta[name]
        return dict(boxsize=m["box"], sgn=m["sgn"], face=m["face"], centre=m["centre"], rcase=m["rcase"], ld=m["ld"],
                    ld2=m["ld2"], nrepperp=m["nrep"], fovradiants=float.fromhex(m["fovradiants"]))


@pytest.fixture(scope="session")
def golden():
    return GoldenCases()


def unhex(v):
    return float.fromhex(v)
