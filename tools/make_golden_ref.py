#!/usr/bin/env python
"""Golden outputs of the reference's own C driver/digestion (oracle/_ref, built by oracle/Makefile.ref where the reference
tree is present) for tests/test_oracle_ref.py and the q_cond test of tests/test_host_emulation.py, so that those
comparisons run without the reference tree.  Symmetric matrices are stored as their lower triangles.
Usage: python tools/make_golden_ref.py   (writes tests/golden/ref_driver_h2o.npz)
"""
import os
import sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
from pyscf_b200 import gto
from oracle import ref_driver as R

H2O = 'O 0 0 0; H 0 -0.757 0.587; H 0 0.757 0.587'
if not R.available():
    sys.exit('oracle/_ref/libcvhf_ref.so is not built (make -C oracle ref)')


def tril(a):
    i, j = np.tril_indices(a.shape[-1])
    return np.ascontiguousarray(a[..., i, j])


out = {}
# test_reference_driver_fingerprints: H2O/cc-pVDZ, random dm (seed 1) with hermi=0, identity with hermi=1
mol = gto.M(atom=H2O, basis='cc-pvdz')
nao = mol.nao
np.random.seed(1)
dm = np.random.random((nao, nao))
out['dz_vj'], out['dz_vk'] = R.get_jk(mol, dm, hermi=0)
vj, vk = R.get_jk(mol, np.eye(nao), hermi=1)
out['dz_eye_vj'], out['dz_eye_vk'] = tril(vj), tril(vk)
# test_reference_driver_equals_oracle_driver: H2O/cc-pVTZ, two symmetrised random dms (seed 4), Coulomb and erf(omega=0.4)
mol = gto.M(atom=H2O, basis='cc-pvtz')
np.random.seed(4)
dm = np.random.random((2, mol.nao, mol.nao))
dm = dm + dm.transpose(0, 2, 1)
for tag, omega in (('tz', None), ('tz_lr', 0.4)):
    vj, vk = R.get_jk(mol, dm, hermi=1, omega=omega)
    out[tag + '_vj'], out[tag + '_vk'] = tril(vj), tril(vk)
# test_q_cond_is_the_reference_bound_for_d_and_f_shells: CVHFnr_int2e_q_cond on a distorted H2O/cc-pVTZ
mol = gto.M(atom='O 0 0 0; H 0 -0.757 0.587; H 0.3 0.757 0.587', basis='cc-pvtz')
out['q_cond_tz'] = R.q_cond(mol)
path = os.path.join(ROOT, 'tests', 'golden', 'ref_driver_h2o.npz')
np.savez_compressed(path, **out)
print(path, os.path.getsize(path), 'bytes')
