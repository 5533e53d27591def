"""The reference's own C driver/digestion (oracle/_ref, fed with the oracle's integral function) agrees with the
oracle's restatement and reproduces the reference fingerprints.  Its outputs are stored in tests/golden/ref_driver_h2o.npz
(tools/make_golden_ref.py), so the comparison runs without the reference tree."""
import os

import numpy as np
import pytest

from pyscf_b200 import gto
from oracle import oracle as O

H2O = 'O 0 0 0; H 0 -0.757 0.587; H 0 0.757 0.587'
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'ref_driver_h2o.npz')


@pytest.fixture(scope='module')
def ref():
    return np.load(GOLDEN)


def test_reference_driver_fingerprints(ref):
    mol = gto.M(atom=H2O, basis='cc-pvdz')
    nao = mol.nao
    np.random.seed(1)
    dm = np.random.random((nao, nao))
    vj, vk = ref['dz_vj'], ref['dz_vk']
    assert abs(np.linalg.norm(vj) - 77.035779188661465) < 1e-9      # pyscf/scf/test/test_rhf.py:908
    assert abs(O.fp(vk) - (-12.365527167710301)) < 1e-9             # :934
    rj, rk = O.get_jk(mol, dm)
    assert abs(vj - rj).max() < 1e-11 and abs(vk - rk).max() < 1e-11
    vj, vk = O.unpack_tril(ref['dz_eye_vj'], nao), O.unpack_tril(ref['dz_eye_vk'], nao)
    assert abs(O.fp(vj) - 1.6593323222866125) < 1e-9 and abs(O.fp(vk) - (-1.4662135224053987)) < 1e-9
    rj, rk = O.get_jk(mol, np.eye(nao))
    assert abs(vj - rj).max() < 1e-11 and abs(vk - rk).max() < 1e-11


def test_reference_driver_equals_oracle_driver(ref):
    mol = gto.M(atom=H2O, basis='cc-pvtz')
    nao = mol.nao
    np.random.seed(4)
    dm = np.random.random((2, nao, nao))
    dm = dm + dm.transpose(0, 2, 1)
    vj, vk = O.unpack_tril(ref['tz_vj'], nao), O.unpack_tril(ref['tz_vk'], nao)
    rj, rk = O.get_jk(mol, dm)
    assert abs(vj - rj).max() < 1e-11 and abs(vk - rk).max() < 1e-11
    vj, vk = O.unpack_tril(ref['tz_lr_vj'], nao), O.unpack_tril(ref['tz_lr_vk'], nao)
    rj, rk = O.get_jk(mol, dm, omega=0.4)
    assert abs(vj - rj).max() < 1e-11 and abs(vk - rk).max() < 1e-11
