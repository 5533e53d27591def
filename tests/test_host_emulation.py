"""CPU tests of the host logic (Mole tables, C-ABI loading, error behaviour) and of the kernel
arithmetic through the CPU SIMT emulation of the CUDA templates (tests/emu/libb200jk_emu.so, built
from the SAME sources with -DB200JK_EMULATE).  The emulation is test infrastructure only."""
import ctypes
import os

import numpy as np
import pytest

from pyscf_b200 import gto, lib as b2lib
from pyscf_b200.gto.mole import geometry, make_auxmol
from pyscf_b200.jk import VHFOpt
from oracle import oracle as O

H2O = 'O 0 0 0; H 0 -0.757 0.587; H 0 0.757 0.587'
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_table_sizes_match_survey():
    # SURVEY.md §8 table: nbas / nao / naux of the benchmark configs
    m = gto.M(atom=H2O, basis='sto-3g')
    assert (m.nbas, m.nao, m.nelectron) == (5, 7, 10)
    m = gto.M(atom=geometry('benzene'), basis='cc-pvtz')
    assert (m.nbas, m.nao, m.nelectron) == (90, 264, 42)
    m = gto.M(atom=geometry('c60'), basis='def2-svp')
    assert (m.nbas, m.nao) == (360, 840)
    aux = make_auxmol(m)
    assert (aux.nbas, aux.nao, int(aux._bas[:, 1].max())) == (1500, 4500, 4)
    m = gto.M(atom=geometry('gly30'), basis='cc-pvdz')       # config 5: C60H92N30O31
    assert (m.natm, m.nbas, m.nao, m.nelectron // 2) == (213, 881, 2154, 455)
    aux = make_auxmol(m)
    assert (aux.nbas, aux.nao) == (3732, 10586)
    m = gto.M(atom=geometry('taxol'), basis='def2-tzvp')     # config 4: C47H51NO14 (tools/make_taxol.py)
    assert (m.natm, m.nbas, m.nao, m.nelectron // 2, int(m._bas[:, 1].max())) == (113, 886, 2228, 226, 3)
    aux = make_auxmol(m)
    assert (aux.nbas, aux.nao, int(aux._bas[:, 1].max())) == (1856, 5598, 4)
    # chemically sane: no two atoms closer than a bond, no non-hydrogen pair closer than 1.19 A (C=O)
    r = m.atom_coords() * 0.52917721092
    d = np.sqrt(((r[:, None] - r[None]) ** 2).sum(-1)) + 10 * np.eye(m.natm)
    heavy = m._atm[:, 0] > 1
    assert d.min() > 0.94 and d[np.ix_(heavy, heavy)].min() > 1.19


def test_env_layout():
    m = gto.M(atom=H2O, basis='sto-3g')
    # pyscf/gto/mole.py:58-88: PTR_ENV_START = 20, coordinates in Bohr
    assert m._atm[0, 1] == 20 and m._atm.shape == (3, 6) and m._bas.shape == (5, 8)
    assert abs(m._env[m._atm[1, 1] + 1] - (-0.757 / 0.52917721092)) < 1e-14
    # gto_norm(0, 1) documented value, pyscf/gto/mole.py:146-147
    from pyscf_b200.gto.mole import gto_norm
    assert abs(gto_norm(0, 1.0) - 2.5264751109842591) < 1e-14


def test_cabi_library_exports_every_symbol():
    path = b2lib.DEFAULT_LIB
    assert os.path.exists(path), 'build the library first (python -c "import __graft_entry__ as g; g.build()")'
    lib = ctypes.CDLL(path)
    hdr = open(os.path.join(ROOT, 'include', 'b200jk.h')).read()
    import re
    declared = sorted(set(re.findall(r'\b(b200jk_[a-z0-9_]+)\s*\(', hdr)))
    assert len(declared) >= 14
    for s in declared:
        assert hasattr(lib, s), s
    lib.b200jk_version.restype = ctypes.c_char_p
    assert b'sm_100a' in lib.b200jk_version()


def test_no_silent_cpu_fallback():
    # without a GPU the product library must fail loudly, never compute on the CPU
    import torch
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    m = gto.M(atom=H2O, basis='sto-3g')
    with pytest.raises(RuntimeError, match='no CUDA device'):
        VHFOpt(m)


@pytest.mark.parametrize('basis', ['sto-3g', '6-31g', 'cc-pvdz'])
def test_emulated_kernels_match_oracle(emu_lib, basis):
    mol = gto.M(atom=H2O, basis=basis)
    nao = mol.nao
    np.random.seed(1)
    dm = np.random.random((nao, nao))
    dm = dm + dm.T
    opt = VHFOpt(mol, libpath=emu_lib)
    vj, vk = opt.get_jk(dm, hermi=1)
    rj, rk = O.get_jk(mol, dm)
    assert abs(vj - rj).max() < 1e-11 and abs(vk - rk).max() < 1e-11
    # hermi=0, two density matrices, leading dims preserved
    dms = np.random.random((2, nao, nao))
    vj, vk = opt.get_jk(dms, hermi=0)
    rj, rk = O.get_jk(mol, dms)
    assert vj.shape == dms.shape and vk.shape == dms.shape
    assert abs(vj - rj).max() < 1e-11 and abs(vk - rk).max() < 1e-11
    # with_j / with_k switches return None for the one not requested (pyscf/scf/hf.py:963)
    vj1, vk1 = opt.get_jk(dm, hermi=1, with_k=False)
    assert vk1 is None and abs(vj1 - O.get_jk(mol, dm)[0]).max() < 1e-11
    vj1, vk1 = opt.get_jk(dm, hermi=1, with_j=False)
    assert vj1 is None


def test_emulated_f_functions_and_fingerprints(emu_lib):
    mol = gto.M(atom='He 0 0 0; Ne 1.2 0.3 0', basis='cc-pvtz')  # f shell on Ne
    nao = mol.nao
    np.random.seed(3)
    dm = np.random.random((nao, nao))
    dm = dm + dm.T
    opt = VHFOpt(mol, libpath=emu_lib)
    vj, vk = opt.get_jk(dm)
    rj, rk = O.get_jk(mol, dm)
    assert abs(vj - rj).max() < 1e-10 and abs(vk - rk).max() < 1e-10


def test_emulated_reference_fingerprints(emu_lib):
    # pyscf/scf/test/test_rhf.py:896-934 through the device code path (emulated)
    mol = gto.M(atom=H2O, basis='cc-pvdz')
    nao = mol.nao
    opt = VHFOpt(mol, libpath=emu_lib)
    np.random.seed(1)
    dm = np.random.random((nao, nao))
    vj, vk = opt.get_jk(dm, hermi=0)
    assert abs(np.linalg.norm(vj) - 77.035779188661465) < 1e-9
    assert abs(O.fp(vk) - (-12.365527167710301)) < 1e-9
    vj, vk = opt.get_jk(np.eye(nao), hermi=1)
    assert abs(O.fp(vj) - 1.6593323222866125) < 1e-9 and abs(O.fp(vk) - (-1.4662135224053987)) < 1e-9
    opt_lr = VHFOpt(mol, omega=1.5, libpath=emu_lib)
    vj, vk = opt_lr.get_jk(dm, hermi=0)
    assert abs(O.fp(vj) - (-10.015956161068031)) < 1e-9 and abs(O.fp(vk) - (-11.399103957754445)) < 1e-9


def test_emulated_screening_and_errors(emu_lib):
    # a stretched molecule: screening must drop quartets without changing J/K beyond the tolerance
    mol = gto.M(atom='O 0 0 0; H 0 -0.757 0.587; H 0 0.757 0.587; O 0 0 12; H 0 -0.757 12.587; H 0 0.757 12.587',
                basis='6-31g')
    nao = mol.nao
    np.random.seed(2)
    dm = np.random.random((nao, nao)) * 1e-2
    dm = dm + dm.T
    opt = VHFOpt(mol, libpath=emu_lib)
    vj, vk = opt.get_jk(dm)
    rj, rk = O.get_jk(mol, dm, screen=False)
    assert abs(vj - rj).max() < 1e-10 and abs(vk - rk).max() < 1e-10
    # a loose threshold must reject quartets on device and stay within the implied error bound
    n_all = opt.stats()['quartets_computed']
    opt2 = VHFOpt(mol, direct_scf_tol=1e-9, libpath=emu_lib)
    vj2, vk2 = opt2.get_jk(dm * 1e-6)
    st = opt2.stats()
    assert st['quartets_screened'] > 0 and st['quartets_computed'] < n_all
    assert abs(vj2 - rj * 1e-6).max() < 1e-7 and abs(vk2 - rk * 1e-6).max() < 1e-7
    with pytest.raises(RuntimeError):
        opt.get_jk(np.zeros((nao + 1, nao + 1)))
    q = opt.q_cond
    qo = O.q_cond(mol)
    big = qo > 1e-12  # negligible pairs are dropped on the device side (reported as the 1e-100 floor)
    assert q.shape == qo.shape and abs(np.log(q[big] / qo[big])).max() < 1e-9  # identical to CVHFnr_int2e_q_cond


def test_q_cond_is_the_reference_bound_for_d_and_f_shells(emu_lib):
    """b200jk_get_q_cond == CVHFnr_int2e_q_cond (pyscf/lib/vhf/optimizer.c:408-454) for every angular momentum: the device
    bounds are over the normalised real-spherical functions, general contractions take the maximum over their segments.
    Checked against the oracle's restatement and against the reference's own C routine (its output stored in
    tests/golden/ref_driver_h2o.npz by tools/make_golden_ref.py)."""
    mol = gto.M(atom='O 0 0 0; H 0 -0.757 0.587; H 0.3 0.757 0.587', basis='cc-pvtz')
    assert int(mol._bas[:, 1].max()) == 3
    opt = VHFOpt(mol, libpath=emu_lib)
    q = opt.q_cond
    qo = O.q_cond(mol)
    assert abs(np.log(q / qo)).max() < 1e-9
    qr = np.load(os.path.join(ROOT, 'tests', 'golden', 'ref_driver_h2o.npz'))['q_cond_tz']
    assert abs(np.log(q / qr)).max() < 1e-9
    # erf-attenuated operator
    opt = VHFOpt(mol, omega=0.4, libpath=emu_lib)
    assert abs(np.log(opt.q_cond / O.q_cond(mol, omega=0.4))).max() < 1e-9


def test_emulated_experimental_layouts(emu_lib, emu_lib_experimental):
    """Primitive batching (QClass::PB) and the part-per-warp lane layout (GroupCfg::PPW) are compile-time options that are
    off in the shipped library until measured; they must give the same J/K as the default layout (same primitive order,
    so only the order of the reductions differs) for d/f shells, hermi 0/1 and the erf / erfc operators."""
    for atom, basis, omega in [(H2O, 'cc-pvdz', None), ('He 0 0 0; Ne 1.2 0.3 0', 'cc-pvtz', None), (H2O, 'cc-pvdz', -0.4),
                               ('O 0 0 0; O 0 0 1.2', 'cc-pvdz', 0.7)]:
        mol = gto.M(atom=atom, basis=basis)
        nao = mol.nao
        np.random.seed(3)
        dms = np.random.random((2, nao, nao))
        a = VHFOpt(mol, omega=omega, libpath=emu_lib_experimental).get_jk(dms, hermi=0)
        b = VHFOpt(mol, omega=omega, libpath=emu_lib).get_jk(dms, hermi=0)
        assert abs(a[0] - b[0]).max() < 1e-11 and abs(a[1] - b[1]).max() < 1e-11
        d = dms[0] + dms[0].T
        a = VHFOpt(mol, omega=omega, libpath=emu_lib_experimental).get_jk(d, hermi=1)
        r = O.get_jk(mol, d, omega=omega)
        assert abs(a[0] - r[0]).max() < 1e-10 and abs(a[1] - r[1]).max() < 1e-10


# ---- boundary semantics (ADVICE round 1): tags, density_fit routing, range-separation from the molecule, cache lifetime
def test_tags_expire_on_arithmetic():
    """lib.tag_array semantics (pyscf/lib/numpy_helper.py:1477-1484): ufunc results and slices carry no orbital tags."""
    from pyscf_b200.df import TaggedDM
    from pyscf_b200.veff import tag_array
    c = np.random.RandomState(0).standard_normal((6, 2))
    dm = TaggedDM(2 * c.dot(c.T), mo_coeff=c, mo_occ=np.array([2.0, 2.0]))
    assert dm.mo_coeff is c
    for derived in (dm - 0.5 * dm, dm * 0.5, dm + dm, -dm, dm[:3], np.asarray(dm) * 1.0):
        assert getattr(derived, 'mo_coeff', None) is None and getattr(derived, 'mo_occ', None) is None
    assert type(dm - dm) is np.ndarray
    v = tag_array(np.eye(3), ecoul=1.5)
    assert v.ecoul == 1.5 and not hasattr(v * 2.0, 'ecoul')


def test_df_get_jk_ignores_stale_tags(emu_lib):
    """DF.get_jk(tagged - other) must equal the untagged result (the stale orbitals are not used)."""
    from pyscf_b200.df import DF, TaggedDM
    mol = gto.M(atom='O 0 0 0; H 0 -0.757 0.587; H 0 0.757 0.587', basis='sto-3g')
    nao = mol.nao
    rng = np.random.RandomState(3)
    c = np.linalg.qr(rng.standard_normal((nao, 3)))[0]
    dm = TaggedDM(2 * c.dot(c.T), mo_coeff=c, mo_occ=np.full(3, 2.0))
    other = rng.standard_normal((nao, nao))
    other = other + other.T
    d = DF(mol, 'weigend', libpath=emu_lib).build()
    vj1, vk1 = d.get_jk(dm - other)
    vj2, vk2 = d.get_jk(np.asarray(dm) - other)
    assert abs(vj1 - vj2).max() < 1e-12 and abs(vk1 - vk2).max() < 1e-12
    vk_tag = d.get_jk(dm)[1]
    assert abs(vk_tag - d.get_jk(np.asarray(dm))[1]).max() < 1e-10   # occupied-orbital path == general path on the tagged density


class _StandInSCF:
    """Minimal stand-in for pyscf.scf.hf.SCF with the reference's call order: get_veff -> get_jk(mol, dm, hermi), get_j/get_k
    funnel into get_jk (pyscf/scf/hf.py:2161-2201); reset(mol) (hf.py:2331)."""
    direct_scf = True
    direct_scf_tol = 1e-13

    def __init__(self, mol):
        self.mol = mol
        self.calls = []
        self._eri = 'incore'
        self.nreset = 0

    def make_rdm1(self):
        return np.eye(self.mol.nao)

    def get_jk(self, mol=None, dm=None, hermi=1, with_j=True, with_k=True, omega=None):
        self.calls.append(('exact', with_j, with_k, omega))
        n = self.mol.nao
        return (np.full((n, n), 1.0) if with_j else None), (np.full((n, n), 2.0) if with_k else None)

    def get_j(self, mol=None, dm=None, hermi=1, omega=None):
        return self.get_jk(mol, dm, hermi, with_k=False, omega=omega)[0]

    def get_k(self, mol=None, dm=None, hermi=1, omega=None):
        return self.get_jk(mol, dm, hermi, with_j=False, omega=omega)[1]

    def get_veff(self, mol=None, dm=None):
        vj, vk = self.get_jk(mol, dm, 1)
        return vj - 0.5 * vk

    def reset(self, mol=None):
        self.nreset += 1
        if mol is not None:
            self.mol = mol
        return self


class _FakeDF:
    def __init__(self):
        self.calls = []
        self.nreset = 0

    def get_jk(self, dm, hermi=1, with_j=True, with_k=True, direct_scf_tol=1e-13, omega=None):
        self.calls.append((with_j, with_k, omega))
        n = np.asarray(dm).shape[-1]
        return (np.full((n, n), 10.0) if with_j else None), (np.full((n, n), 20.0) if with_k else None)

    def reset(self, mol=None):
        self.nreset += 1


def test_density_fit_routes_like_dfhf():
    """density_fit(mf) returns a (_DFHF, mf.__class__) object whose get_jk is served by with_df (pyscf/df/df_jk.py:104-179)."""
    from pyscf_b200.df import density_fit, _DFHF
    mol = gto.M(atom='O 0 0 0; H 0 -0.757 0.587; H 0 0.757 0.587', basis='sto-3g')
    mf = _StandInSCF(mol)
    fake = _FakeDF()
    dfmf = density_fit(mf, with_df=fake)
    assert isinstance(dfmf, _DFHF) and isinstance(dfmf, _StandInSCF) and type(dfmf).__name__ == 'DF_StandInSCF'
    assert dfmf._eri is None and not dfmf.direct_scf and dfmf.with_df is fake
    dm = np.eye(mol.nao)
    vj, vk = dfmf.get_jk(mol, dm)
    assert vj[0, 0] == 10.0 and vk[0, 0] == 20.0 and fake.calls[-1] == (True, True, None)
    assert dfmf.get_veff(mol, dm)[0, 0] == 0.0                         # get_veff funnels into the DF get_jk
    assert dfmf.get_k(mol, dm, omega=0.3)[0, 0] == 20.0 and fake.calls[-1] == (False, True, 0.3)
    # only_dfj: J fitted, K from the class's exact get_jk; direct_scf switched back on (df_jk.py:133-137,157-179)
    dfmf2 = density_fit(mf, with_df=fake, only_dfj=True)
    vj, vk = dfmf2.get_jk(mol, dm)
    assert vj[0, 0] == 10.0 and vk[0, 0] == 2.0 and dfmf2.direct_scf
    assert fake.calls[-1] == (True, False, None) and dfmf2.calls[-1] == ('exact', False, True, None)
    # with_df = None switches density fitting off (df_jk.py:153-154)
    dfmf.with_df = None
    assert dfmf.get_jk(mol, dm)[0][0, 0] == 1.0
    dfmf.with_df = fake
    dfmf.reset()
    assert fake.nreset == 1 and dfmf.nreset == 1
    # an object patched with jk.patch keeps the B200 4-center builder as its exact path
    marker = []

    def inst_get_jk(mol=None, dm=None, hermi=1, with_j=True, with_k=True, omega=None):
        marker.append((with_j, with_k))
        return None, np.full((mol.nao, mol.nao), 7.0)
    mf2 = _StandInSCF(mol)
    mf2.get_jk = inst_get_jk
    dfmf3 = density_fit(mf2, with_df=fake, only_dfj=True)
    assert dfmf3.get_jk(mol, dm)[1][0, 0] == 7.0 and marker == [(False, True)]


def test_omega_none_uses_the_molecules_operator(emu_lib):
    """omega=None means the molecule's own range separation (pyscf/scf/hf.py:1021, pyscf/gto/mole.py:2940-2951)."""
    from pyscf_b200 import jk as JK
    from pyscf_b200.df import DF
    mol = gto.M(atom='O 0 0 0; H 0 -0.757 0.587; H 0 0.757 0.587', basis='sto-3g')
    np.random.seed(2)
    dm = np.random.random((mol.nao,) * 2)
    dm = dm + dm.T
    full = JK.VHFOpt(mol, libpath=emu_lib).get_jk(dm)
    lr = JK.VHFOpt(mol, omega=0.3, libpath=emu_lib).get_jk(dm)
    assert abs(full[1] - lr[1]).max() > 1e-3
    with mol.with_range_coulomb(0.3):
        inside = JK.VHFOpt(mol, libpath=emu_lib).get_jk(dm)
        assert JK.effective_omega(mol, None) == 0.3 and JK.effective_omega(mol, 0.0) == 0.0
        d_in = DF(mol, 'weigend', libpath=emu_lib)
        kin = d_in.get_jk(dm)[1]
    assert abs(inside[0] - lr[0]).max() < 1e-12 and abs(inside[1] - lr[1]).max() < 1e-12
    assert JK.effective_omega(mol, None) == 0.0
    kfull = DF(mol, 'weigend', libpath=emu_lib).get_jk(dm)[1]
    klr = DF(mol, 'weigend', libpath=emu_lib).get_jk(dm, omega=0.3)[1]
    assert abs(kin - klr).max() < 1e-12 and abs(kin - kfull).max() > 1e-3
    # a tensor built for one operator is not reused when the molecule's operator changes
    d = DF(mol, 'weigend', libpath=emu_lib)
    k0 = d.get_jk(dm)[1]
    with mol.with_range_coulomb(0.3):
        k1 = d.get_jk(dm)[1]
    assert abs(k0 - kfull).max() < 1e-12 and abs(k1 - klr).max() < 1e-12


def test_patch_cache_follows_the_molecule(emu_lib):
    """jk.patch: optimizers are dropped by mf.reset() and rebuilt when the molecule's tables change in place."""
    from pyscf_b200 import jk as JK
    mol = gto.M(atom='O 0 0 0; H 0 -0.757 0.587; H 0 0.757 0.587', basis='sto-3g')
    mf = JK.patch(_StandInSCF(mol), libpath=emu_lib)
    dm = np.eye(mol.nao)
    k0 = mf.get_jk(mol, dm)[1]
    opt0 = mf._b200_opts.get(mol, None, libpath=emu_lib)
    assert mf._b200_opts.get(mol, None, libpath=emu_lib) is opt0          # cached
    mol._env[mol._atm[1, 1] + 2] += 0.2                               # move an atom in place (set_geom_-like)
    k1 = mf.get_jk(mol, dm)[1]
    assert abs(k1 - k0).max() > 1e-4 and mf._b200_opts.get(mol, None, libpath=emu_lib) is not opt0
    mf.reset()
    assert mf.nreset == 1 and not mf._b200_opts._d
    # the module-level cache is bounded and keyed on live objects
    JK._opt_cache.clear()


def test_long_ket_ranges_walk_sub_chunks(emu_lib):
    """A CTA whose ket range is longer than the shared ket list (KCH_MAX = 512) walks it in sub-chunks with the stationary J[ij]
    block kept in registers: forced here with one CTA per bra pair (B200JK_WANT_CTAS=1, read once per process, hence the
    subprocess) on (Gly)4/STO-3G, whose 1176 (ss| pairs need three sub-chunks; hermi 1 and a stack of non-symmetric densities."""
    import subprocess, sys, os, textwrap
    code = textwrap.dedent('''
        import os, sys, numpy as np
        sys.path.insert(0, %r)
        from pyscf_b200 import gto
        from pyscf_b200.gto.mole import geometry
        from pyscf_b200.jk import VHFOpt
        from oracle import oracle as O
        mol = gto.M(atom=geometry('gly4'), basis='sto-3g')
        nao = mol.nao
        np.random.seed(2)
        dm = np.random.random((nao, nao)) * 0.1
        opt = VHFOpt(mol, libpath=%r)
        for d, hermi in ((dm + dm.T, 1), (np.array([dm, dm.T * 0.5]), 0)):
            vj, vk = opt.get_jk(d, hermi=hermi)
            rj, rk = O.get_jk(mol, d)
            assert abs(vj - rj).max() < 1e-10 and abs(vk - rk).max() < 1e-10
        print('OK')
    ''') % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), emu_lib)
    env = dict(os.environ, B200JK_WANT_CTAS='1')
    out = subprocess.run([sys.executable, '-c', code], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and 'OK' in out.stdout, out.stderr[-2000:]
