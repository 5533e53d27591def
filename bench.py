#!/usr/bin/env python
"""bench.py — J/K Fock-build seconds per SCF iteration (BASELINE.json metric) on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--no-df] [--dump-outputs DIR]

A "step" = one J/K Fock build (one get_jk-equivalent call) for the workload's density matrix.
Headline workload (the top-level value / e2e / roofline of the JSON line): configs[1] of BASELINE.json, benzene / cc-pVTZ RHF,
4-center direct J/K.  The SAME JSON line carries, under "df", one full record (value, e2e, roofline with per-stage figures,
parity) for every density-fitting configuration of BASELINE.json that fits the N GPUs of the run:
    c60-def2svp-df            configs[2]  (N >= 1)
    taxol-def2tzvp-df         configs[3]  (N >= 1: the 111 GB tensor fits one 180 GB B200; sharded by auxiliary rows for N > 1)
    gly30-ccpvdz-df-wb97x     configs[4]  (N >= 4: omega-B97X needs get_jk on the Coulomb tensor AND get_k(omega=0.3) on a second,
                                           erf-attenuated tensor, 2 x 196.6 GB)
Each DF record is measured by a child process per rank (own NCCL group on another port), so that a failure or a hang in one
configuration cannot take the headline number down with it; a per-record timeout bounds the whole run.

Timed numbers (headline and every DF record)
  value / ms_per_step : J/K build with D, (C_occ,) J, K resident in HBM, CUDA events per step on the launching stream,
                        256 MiB L2 flush between steps outside the event pairs; N > 1: one build sharded over the ranks
                        (bra shell-pair batches / auxiliary rows) + ONE NCCL all-reduce of [J;K] inside the timed region,
                        max over ranks.
  e2e                 : the same build through the public plugin call (VHFOpt.get_jk / DF.get_jk / ShardedJK.get_jk) with pinned
                        HOST buffers (H2D of D, C_occ and D2H of J,K inside the timed region).
  roofline            : direct: all class launches of one build against the measured FP64 FMA-pipe peak (b200jk_fp64_peak).
                        DF: the dominant kernel (stage 1 of DF-K, tcgen05 int8 slices) per launch from CUDA events the library
                        records around every launch, against 2 x the measured bf16 tensor peak; other stages listed beside it.
  parity              : max |dJ|, |dK| of the (all-reduced) result against oracle-made golden vectors (tests/golden) on the
                        reference's own parity density (seed 1), at every N.
  cpu_baseline        : rank 0, N = 1 only.
--impl reference times the CPU arm alone with the same JSON schema: the reference's own driver/screening/digestion C
(oracle/_ref, compiled from /root/reference/pyscf/lib/vhf) around the oracle's integral function; every step is a bounded
sample (every m-th surviving shell quartet per thread, time x m).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the benchmark leaves the source tree as it found it (it may be read-only)

import numpy as np  # noqa: E402

WORKLOADS = {
    'benzene-ccpvtz-direct': dict(geom='benzene', basis='cc-pvtz', nocc=21, kind='direct'),
    'benzene-ccpvdz-direct': dict(geom='benzene', basis='cc-pvdz', nocc=21, kind='direct'),
    'h2o-ccpvdz-direct': dict(geom='h2o', basis='cc-pvdz', nocc=5, kind='direct'),
    'c60-def2svp-df': dict(geom='c60', basis='def2-svp', nocc=180, kind='df'),                  # BASELINE configs[2]
    'benzene-def2svp-df': dict(geom='benzene', basis='def2-svp', nocc=21, kind='df'),
    'gly30-ccpvdz-df': dict(geom='gly30', basis='cc-pvdz', nocc=455, kind='df'),               # full-range part of configs[4]
    'gly30-ccpvdz-df-wb97x': dict(geom='gly30', basis='cc-pvdz', nocc=455, kind='df', omega=0.3),   # BASELINE configs[4]
    'taxol-def2tzvp-df': dict(geom='taxol', basis='def2-tzvp', nocc=226, kind='df'),           # BASELINE configs[3]
    'gly4-ccpvdz-df': dict(geom='gly4', basis='cc-pvdz', nocc=65, kind='df'),
    'gly4-ccpvdz-df-wb97x': dict(geom='gly4', basis='cc-pvdz', nocc=65, kind='df', omega=0.3),
}
# DF records appended to the headline line, timed with the run's --steps / --warmup: (workload, smallest N it fits,
# child timeout in seconds)
DF_EXTRAS = [('c60-def2svp-df', 1, 240), ('taxol-def2tzvp-df', 1, 300), ('gly30-ccpvdz-df-wb97x', 4, 300)]
TENSOR_GB = {'taxol-def2tzvp-df': 111.2, 'gly30-ccpvdz-df-wb97x': 2 * 196.6, 'c60-def2svp-df': 12.7}


def scf_like_dm(nao, nocc, seed=1):
    rng = np.random.RandomState(seed)
    c, _ = np.linalg.qr(rng.standard_normal((nao, nocc)))
    return 2.0 * c.dot(c.T)


def parity_dm(nao):
    np.random.seed(1)    # the reference's own test idiom (pyscf/scf/test/test_rhf.py:897-899); tools/make_golden.py
    dm = np.random.random((nao, nao))
    return dm + dm.T


def build_mol(w):
    from pyscf_b200 import gto
    from pyscf_b200.gto.mole import geometry
    return gto.M(atom=geometry(w['geom']), basis=w['basis'])


def host_threads():
    """Threads the CPU arms may use: all cores of the box (torchrun exports OMP_NUM_THREADS=1, which must not leak in)."""
    return os.cpu_count() or 1


def cpu_model():
    try:
        for line in open('/proc/cpuinfo'):
            if line.startswith('model name'):
                return line.split(':', 1)[1].strip()
    except Exception:
        pass
    return ''


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region."""

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = False
        self.proc = None

    def run(self):
        q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q,
                                          '--format=csv,noheader,nounits', '-lms', '100'], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.samples.append([t.strip() for t in line.split(',')])
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc:
            try:
                self.proc.terminate()
            except Exception:
                pass
        sm, mx, reasons = [], 0, set()
        for s in self.samples:
            try:
                sm.append(float(s[0]))
                mx = max(mx, float(s[1]))
                for name, v in zip(['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'], s[2:6]):
                    if v.lower().startswith('active'):
                        reasons.add(name)
            except Exception:
                continue
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': mx or None, 'reasons': sorted(reasons),
                'samples': len(sm)}


def algorithmic_bytes(opt):
    """Algorithmic HBM bytes of one direct build (DESIGN.md §4.1): D, J and K once each (3 n^2 doubles) plus the shell-pair
    records the kernels stream (48 B of each 64-byte record are payload)."""
    st = opt.stats()
    n = st['n_sph']
    return 3 * n * n * 8 + st['n_pairs'] * 48


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of `kernel` from the committed `ncu --set full` summary of the
    C60 bench command (profiles/r02_ncu_summary.txt); None when the profile is not there."""
    try:
        tot, on = 0.0, False
        for line in open(os.path.join(ROOT, 'profiles', 'r02_ncu_summary.txt')):
            if line.startswith('kernel:'):
                on = kernel in line
            elif on and ('dram__bytes_read.sum' in line or 'dram__bytes_write.sum' in line):
                f = line.split()
                scale = {'byte': 1.0, 'Kbyte': 1e3, 'Mbyte': 1e6, 'Gbyte': 1e9, 'Tbyte': 1e12}.get(f[2] if len(f) > 2 else 'byte', 1.0)
                tot += float(f[1]) * scale
        return tot or None
    except Exception:
        return None


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        return {}


# ------------------------------------------------------------------------------------------------------------------
def golden_parity(workload, vj, vk, what):
    """max-abs deviation of J/K from the oracle-made golden vectors of this workload (tests/golden), None when there is no
    fixture.  Full matrices for benzene (tools/make_golden.py), sampled elements + fingerprints for the DF configurations
    (tools/make_golden_df_size.py)."""
    name = {'benzene-ccpvtz-direct': 'jk_bz_tz.npz', 'benzene-ccpvdz-direct': 'jk_bz_dz.npz',
            'c60-def2svp-df': 'df_c60_jk.npz', 'gly4-ccpvdz-df': None}.get(workload)
    if not name:
        return None
    path = os.path.join(ROOT, 'tests', 'golden', name)
    if not os.path.exists(path):
        return None
    z = np.load(path)
    if 'idx' in z:      # sampled elements [n, 2] of the oracle's J/K for the density `what`
        key = {'parity': 'p', 'scf': 's'}[what]
        if 'vj_' + key not in z:
            return None
        i, j = z['idx'][:, 0], z['idx'][:, 1]
        return {'max_abs_dJ': float(abs(vj[i, j] - z['vj_' + key]).max()), 'max_abs_dK': float(abs(vk[i, j] - z['vk_' + key]).max()),
                'against': 'tests/golden/%s (%d sampled elements of the CPU oracle J/K)' % (name, len(i)), 'bar': 1e-9}
    if what != 'parity':
        return None
    return {'max_abs_dJ': float(abs(vj - z['vj']).max()), 'max_abs_dK': float(abs(vk - z['vk']).max()),
            'against': 'tests/golden/%s (full J/K of the CPU oracle)' % name, 'bar': 1e-9}


SIZE_FIXTURE = {'c60-def2svp-df': ('c60', None), 'taxol-def2tzvp-df': ('taxol', None), 'gly30-ccpvdz-df': ('gly30', None),
                'gly30-ccpvdz-df-wb97x': ('gly30', 'gly30_lr'), 'gly4-ccpvdz-df': ('gly4', None), 'gly4-ccpvdz-df-wb97x': ('gly4', None)}


def df_size_parity(workload, eng, eng2, step_device, out_d, res_dev, dev, rank, world, dist):
    """Oracle parity of a DF configuration AT ITS SIZE, at every N (fixtures: tools/make_golden_df_size.py, tests/golden/df_size_*):
    sampled tensor columns over the auxiliary rows of every rank, and J/K of the fixture's slab density through BOTH K engines
    (orbital-tagged: tcgen05 occupied-orbital algorithm; bare matrix: general-density algorithm), all-reduced like a timed step."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    import df_size_check as S
    names = SIZE_FIXTURE.get(workload)
    z = S.load(names[0]) if names else None
    if z is None:
        return None
    out = {'against': 'tests/golden/df_size_%s.npz (CPU oracle: %d tensor columns over all auxiliary rows; J rows and K of a density '
                      'supported on %d AOs)' % (names[0], len(z['cols']), len(z['sao'])), 'bar': 1e-9}
    dc = S.check_columns(eng, z)
    if world > 1:
        t = torch.tensor([dc if dc is not None else -1.0], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dc = float(t[0])
    out['max_abs_dcderi_cols'] = dc
    c = S.slab_coeff(z)
    dm_t = torch.from_numpy(2.0 * c.dot(c.T)).to(dev)
    occ_t = torch.from_numpy(np.ascontiguousarray(c * np.sqrt(2.0))).to(dev)
    z2 = S.load(names[1]) if (names[1] and eng2 is not None) else None
    for tag, occ in (('orbital_tagged', occ_t), ('general_density', None)):
        step_device(dm_t, occ, c.shape[1] if occ is not None else 0)
        torch.cuda.synchronize()
        r = out_d.cpu().numpy()
        rec = S.compare_jk(z, r[0], r[1])
        if z2 is not None:      # K of the erf-attenuated tensor (get_k(omega)), same slab density
            rec['long_range_K'] = S.compare_jk(z2, None, r[2])
        out[tag] = rec
    # the timed SCF-like density: tensor-core engine (the timed result) against the general-density engine on the same tensor
    step_device(occ_t=None, nocc=0)
    torch.cuda.synchronize()
    r = out_d.cpu().numpy()
    out['scf_like_density_engines_max_abs_dK'] = float(abs(r[1:] - res_dev[1:]).max())
    out['scf_like_density_engines_max_abs_dJ'] = float(abs(r[0] - res_dev[0]).max())
    return out


DUMP_MAX_ELEMENTS = 1 << 20      # per array: 8 MB of float64; every record of an 8-GPU run stays below 64 MB in all


def dump_outputs(dirname, workload, res):
    """J, K (and K of the erf-attenuated tensor) of the last timed step as <dirname>/<workload>_{J,K,K_omega}.npy, float64.
    A matrix with more than DUMP_MAX_ELEMENTS elements is stored as a fixed sample of its rows (RandomState(0), sorted), so
    that two builds run with the same arguments can be compared element for element."""
    os.makedirs(dirname, exist_ok=True)
    nao = res.shape[-1]
    rows = np.arange(nao)
    if nao * nao > DUMP_MAX_ELEMENTS:
        rows = np.sort(np.random.RandomState(0).choice(nao, DUMP_MAX_ELEMENTS // nao, replace=False))
    for name, a in zip(('J', 'K', 'K_omega'), res):
        np.save(os.path.join(dirname, '%s_%s.npy' % (workload, name)), np.ascontiguousarray(a[rows], dtype=np.float64))


def measure(args, rank, world, dist):
    """One workload on this process group: returns the record (rank 0) or None (other ranks)."""
    import torch
    import ctypes
    from pyscf_b200.jk import VHFOpt
    from pyscf_b200.df import DF, TaggedDM
    w = WORKLOADS[args.workload]
    is_df = w['kind'] == 'df'
    omega2 = w.get('omega')          # second, erf-attenuated tensor + get_k(omega) in every step (range-separated hybrid)
    local = int(os.environ.get('LOCAL_RANK', rank))
    dev = torch.device('cuda', local)
    mol = build_mol(w)
    nao = mol.nao
    rng = np.random.RandomState(1)
    c_occ, _ = np.linalg.qr(rng.standard_normal((nao, w['nocc'])))
    dm_h = 2.0 * c_occ.dot(c_occ.T)
    occ_h = np.ascontiguousarray(c_occ * np.sqrt(2.0))
    t0 = time.time()
    eng2 = h2 = None
    if is_df:
        eng = DF(mol, device=local, shard=(rank, world) if world > 1 else None).build()
        h = eng._handle
        if omega2:
            eng2 = eng.range_coulomb(omega2)
            h2 = eng2._handle
    else:
        eng = VHFOpt(mol, direct_scf_tol=1e-13, device=local)
        h = eng.handle
    torch.cuda.synchronize()
    setup_s = time.time() - t0
    # strong scaling: ONE Fock build is split over the ranks (shell-pair batches / auxiliary rows), partial J,K
    # are summed by a single NCCL all-reduce per build
    handles = [h] + ([h2] if h2 is not None else [])
    stream = torch.cuda.current_stream(dev)
    for hh in handles:
        hh.check(hh.lib.b200jk_set_shard(hh._h, rank, world), 'b200jk_set_shard')
        hh.lib.b200jk_set_stream(hh._h, ctypes.c_void_p(stream.cuda_stream))

    if not is_df and world > 1:
        # measured class times of one unsharded build as the cost table of the multi-GPU partition (rank 0's table on every rank)
        from pyscf_b200.parallel import calibrate_partition
        h.lib.b200jk_set_stream(h._h, None)
        calibrate_partition(h, dm_h[None], rank, world)
        h.lib.b200jk_set_stream(h._h, ctypes.c_void_p(stream.cuda_stream))
    nout = 3 if omega2 else 2
    dm_d = torch.from_numpy(dm_h).to(dev)
    occ_d = torch.from_numpy(occ_h).to(dev)
    out_d = torch.zeros((nout, nao, nao), dtype=torch.float64, device=dev)
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=dev)
    vp = ctypes.c_void_p

    def step_device(dm_t=dm_d, occ_t=occ_d, nocc=w['nocc']):
        if is_df:
            rc = h.lib.b200jk_df_jk_device(h._h, vp(dm_t.data_ptr()), 1, nao, vp(occ_t.data_ptr()) if occ_t is not None else None,
                                           nocc, 1, vp(out_d[0].data_ptr()), vp(out_d[1].data_ptr()))
            h.check(rc, 'b200jk_df_jk_device')
            if omega2:   # vklr = get_k(dm, omega) on the attenuated tensor (pyscf/dft/rks.py:123-127)
                rc = h2.lib.b200jk_df_jk_device(h2._h, vp(dm_t.data_ptr()), 1, nao, vp(occ_t.data_ptr()) if occ_t is not None else None,
                                                nocc, 1, None, vp(out_d[2].data_ptr()))
                h2.check(rc, 'b200jk_df_jk_device(omega)')
        else:
            rc = h.lib.b200jk_direct_jk_device(h._h, vp(dm_t.data_ptr()), 1, nao, 1, vp(out_d[0].data_ptr()), vp(out_d[1].data_ptr()))
            h.check(rc, 'b200jk_direct_jk_device')
        if world > 1:
            dist.all_reduce(out_d)

    for _ in range(args.warmup):
        step_device()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    kern_ms, stage_log, stage_log2 = [], [], []
    launches = 0
    torch.cuda.synchronize()
    t_wall0 = time.time()
    for k in range(args.steps):
        flush.zero_()
        if world > 1:
            dist.barrier()
        evs[k][0].record(stream)
        step_device()
        evs[k][1].record(stream)
        torch.cuda.synchronize()
        km = 0.0
        for hh in handles:
            st = hh.stats()
            km += st['ms_kernels']
            launches += st['kernel_launches']
        kern_ms.append(km)
        if is_df:
            stage_log.append(h.df_stage_times())
            if h2 is not None:
                stage_log2.append(h2.df_stage_times())
    torch.cuda.synchronize()
    t_wall = time.time() - t_wall0
    step_ms = [a.elapsed_time(b) for a, b in evs]
    ms_per_step = float(np.mean(step_ms))
    res_dev = out_d.cpu().numpy().copy()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, args.workload, res_dev)
    # ---- parity on the reference's own test density (seed 1, D + D^T; general-density path for DF) against the oracle golden
    par = None
    try:
        if is_df:
            par = df_size_parity(args.workload, eng, eng2, step_device, out_d, res_dev, dev, rank, world, dist)
        else:
            pd_h = parity_dm(nao)
            step_device(torch.from_numpy(pd_h).to(dev), None, 0)
            torch.cuda.synchronize()
            pr = out_d.cpu().numpy()
            par = golden_parity(args.workload, pr[0], pr[1], 'parity')
    except Exception as e:   # a failed parity leg must be visible, not fatal for the timing record
        par = {'error': repr(e)[:300]}
    # ---- end-to-end through the public plugin call with pinned host buffers (H2D + D2H inside the timed region)
    dm_pin = torch.from_numpy(dm_h).pin_memory().numpy()
    if is_df:
        dm_pub = TaggedDM(dm_pin, mo_coeff=c_occ, mo_occ=np.full(w['nocc'], 2.0))
    else:
        dm_pub = dm_pin
    for hh in handles:
        hh.lib.b200jk_set_stream(hh._h, None)
    sj = sj2 = None
    if world > 1:
        from pyscf_b200.parallel import ShardedJK
        sj = ShardedJK(eng, rank, world)
        sj2 = ShardedJK(eng2, rank, world) if eng2 is not None else None

    def step_public():
        if world > 1:
            vj, vk = sj.get_jk(dm_pub, hermi=1)
            vk2 = sj2.get_jk(dm_pub, hermi=1, with_j=False)[1] if sj2 is not None else None
        else:
            vj, vk = eng.get_jk(dm_pub, hermi=1)
            vk2 = eng.get_jk(dm_pub, hermi=1, with_j=False, omega=omega2)[1] if omega2 else None
        return vj, vk, vk2

    for _ in range(2):
        step_public()
    e2e_ms = []
    for k in range(args.steps):
        flush.zero_()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t = time.perf_counter()
        vj, vk, vk2 = step_public()
        e2e_ms.append((time.perf_counter() - t) * 1e3)
    clocks = sampler.finish()
    e2e_ms_mean = float(np.mean(e2e_ms))
    kernel_ms = float(np.mean(kern_ms))
    rank_ms = None
    if world > 1:
        tt = torch.tensor([ms_per_step, e2e_ms_mean], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_per_step, e2e_ms_mean = float(tt[0]), float(tt[1])
        gk = torch.zeros(world, device=dev, dtype=torch.float64)
        gk[rank] = kernel_ms
        dist.all_reduce(gk)
        rank_ms = [float(x) for x in gk.cpu()]
    if rank != 0:
        for hh in handles:
            hh.close()
        return None
    # ---- roofline
    peaks = load_peaks()
    hbm_peak = peaks.get('hbm_gbs', 6650.0)
    if not is_df:
        from pyscf_b200.flops import direct_jk_flops
        peak = ctypes.c_double(0)
        h.lib.b200jk_fp64_peak(h._h, ctypes.byref(peak))
        flops, n_eri = direct_jk_flops(mol)
        bytes_alg = algorithmic_bytes(eng)
        fp64_ach = flops / world / (kernel_ms * 1e-3) / 1e12
        roof = {'bound': 'fp64', 'achieved': fp64_ach, 'peak': peak.value, 'unit': 'TFLOP/s',
                'frac': fp64_ach / peak.value if peak.value else None, 'traffic': None,
                'kernel': 'jk_class_kernel / jk_tpq_kernel <QClass<LI,LJ,LK,LL,NP>> (all class launches of one build)',
                'kernel_ms_per_step': kernel_ms, 'alg_flops_per_step': flops, 'alg_cart_eris_per_step': n_eri,
                'peak_source': 'b200jk_fp64_peak DFMA micro-benchmark (MEASURED_PEAKS.json has no fp64 entry)',
                'hbm': {'bound': 'hbm', 'achieved': bytes_alg / (kernel_ms * 1e-3) / 1e9, 'peak': hbm_peak, 'unit': 'GB/s',
                        'frac': bytes_alg / (kernel_ms * 1e-3) / 1e9 / hbm_peak, 'alg_bytes_per_step': bytes_alg,
                        'peak_source': 'MEASURED_PEAKS.json hbm_gbs (of measured)' if peaks else 'fallback 6650'}}
        path = '4-center direct J/K (hermi=1, with_j, with_k)'
    else:
        naux = eng.get_naoaux()
        ns = eng.k_slices
        nsl = ns * (ns + 1) // 2                                   # slice GEMMs actually executed (k + l < ns)
        naux2 = eng2.get_naoaux() if eng2 is not None else 0         # rows of the erf-attenuated tensor (fewer: eigenvalue cut of its metric)
        fp64_flops = 4.0 * (naux + naux2) * nao * nao * w['nocc']    # dsymm + dgemm count of the reference (SURVEY §8d), summed over the K builds
        int8_ops = fp64_flops * nsl
        bf16_peak = peaks.get('bf16_tflops_sustained', 1400.0)
        tensor_peak = 2 * bf16_peak
        cderi_bytes = naux * nao * (nao + 1) / 2 * 8

        def mean_stage(log):
            return {k: (float(np.mean([t[k][0] for t in log])), int(log[0][k][1])) for k in log[0]}
        stg = mean_stage(stage_log)
        if stage_log2:
            s2 = mean_stage(stage_log2)
            stg = {k: (stg[k][0] + s2[k][0], stg[k][1] + s2[k][1]) for k in stg}
        half_ops = int8_ops / 2 / world                            # each GEMM stage carries half of the 4*naux*nao^2*nocc count
        stages = {}
        for k in ('k_gemm1', 'k_gemm2'):
            ms_k, n_k = stg[k]
            if n_k:
                stages[k] = {'kernel': 'i8gemm_ar_kernel (stage 1: Y = A C~)' if k == 'k_gemm1' else 'i8gemm_ar_kernel (stage 2: K += Y Y^T, accumulate mode)', 'bound': 'tensor',
                             'launches_per_step': n_k, 'ms_per_launch': ms_k / n_k, 'ms_per_step': ms_k,
                             'alg_int8_ops_per_launch': half_ops / n_k, 'achieved': half_ops / (ms_k * 1e-3) / 1e12,
                             'peak': tensor_peak, 'unit': 'TOP/s (int8)', 'frac': half_ops / (ms_k * 1e-3) / 1e12 / tensor_peak}
                if k == 'k_gemm2':
                    # the kernel computes only the 128 x 64 tiles that touch the upper triangle of the symmetric product
                    mt_, nt_ = (nao + 127) // 128, (nao + 63) // 64
                    done = sum(max(0, nt_ - 2 * a) for a in range(mt_))
                    fexec = done * 128.0 * 64.0 / (nao * nao)
                    stages[k].update({'executed_frac_of_alg_ops': fexec, 'achieved_executed': stages[k]['achieved'] * fexec,
                                      'frac_executed': stages[k]['frac'] * fexec,
                                      'note': 'algorithmic count = the full Y Y^T product of the reference dgemm (SURVEY 8d); the kernel executes '
                                              'only the tiles touching the upper triangle (executed_frac_of_alg_ops, padding included): '
                                              'frac_executed is the tensor-pipe figure, frac the algorithmic one'})
        for k in ('j_rho', 'j_acc'):
            ms_k, n_k = stg.get(k, (0.0, 0))
            if n_k:
                stages[k] = {'kernel': {'j_rho': 'dfj_rho_kernel', 'j_acc': 'dfj_acc_kernel'}[k], 'bound': 'hbm',
                             'launches_per_step': n_k, 'ms_per_step': ms_k, 'alg_bytes_per_step': cderi_bytes / world,
                             'achieved': cderi_bytes / world / (ms_k * 1e-3) / 1e9, 'peak': hbm_peak, 'unit': 'GB/s',
                             'frac': cderi_bytes / world / (ms_k * 1e-3) / 1e9 / hbm_peak}
        ms_k, n_k = stg['k_slice']
        stages['k_slice'] = {'kernel': 'rowmax_kernel + split_long_kernel (int8 slicing of Y)', 'ms_per_step': ms_k,
                             'launches_per_step': n_k}
        ach = int8_ops / world / (kernel_ms * 1e-3) / 1e12
        g1 = stages.get('k_gemm1')
        if g1:     # the dominant kernel: stage 1 of DF-K
            roof = {'bound': 'tensor', 'achieved': g1['achieved'], 'peak': tensor_peak, 'unit': 'TOP/s (int8)', 'frac': g1['frac'],
                    'traffic': ncu_traffic('i8gemm_ar_kernel') if args.workload == 'c60-def2svp-df' and world == 1 else None,
                    'kernel': 'i8gemm_ar_kernel (tcgen05.mma.kind::i8, stage 1 of DF-K: Y = (P|mu nu) C~), CUDA events around '
                              'each of its launches inside the timed steps',
                    'ms_per_launch': g1['ms_per_launch'], 'launches_per_step': g1['launches_per_step'],
                    'alg_int8_ops_per_launch': g1['alg_int8_ops_per_launch']}
        else:
            roof = {'bound': 'tensor', 'achieved': ach, 'peak': tensor_peak, 'unit': 'TOP/s (int8)', 'frac': ach / tensor_peak,
                    'traffic': None, 'kernel': 'whole DF J+K build'}
        roof.update({
                'slice_gemms': nsl, 'stages': stages,
                'whole_build': {'ms_per_step': kernel_ms, 'achieved': ach, 'frac': ach / tensor_peak, 'unit': 'TOP/s (int8)',
                                'note': 'all int8 slice-GEMM work over the whole DF J+K build time (J passes, slicing, both GEMM stages)',
                                'fp64_equiv_flops_per_step': fp64_flops,
                                'fp64_equiv_tflops': fp64_flops / world / (kernel_ms * 1e-3) / 1e12},
                'peak_source': 'tensor: 2 x MEASURED_PEAKS.json bf16_tflops_sustained (int8 dense = 2x bf16 on sm_100a; sustained '
                               'because the kernel runs inside a long step); hbm: MEASURED_PEAKS.json hbm_gbs'
                               if peaks else 'fallback 2 x 1400 TFLOP/s, 6650 GB/s (B200_PROFILING.md)'})
        path = 'DF J/K (cderi resident, K via tcgen05 int8 slices, %d slices)' % ns
        if omega2:
            path += ' + get_k(omega=%g) on the erf-attenuated tensor (omega-B97X, pyscf/dft/rks.py:123-127)' % omega2
    # ---- CPU baseline (oracle port), rank 0, N=1 only
    cpu = None
    if world == 1 and not args.no_cpu:
        try:
            if is_df:
                cpu = cpu_baseline_df(mol, dm_h, c_occ, args.workload)
            else:
                cpu = cpu_baseline(mol, dm_h, args.workload)
            if cpu.get('vj') is not None:
                cpu['max_abs_dJ_vs_gpu'] = float(abs(vj - cpu.pop('vj')).max())
                cpu['max_abs_dK_vs_gpu'] = float(abs(vk - cpu.pop('vk')).max())
        except Exception as e:
            cpu = {'error': repr(e)[:300]}
    dev_vs_pub = max(abs(vj - res_dev[0]).max(), abs(vk - res_dev[1]).max())
    if vk2 is not None:
        dev_vs_pub = max(dev_vs_pub, abs(vk2 - res_dev[2]).max())
    h2d = nao * nao * 8 + (nao * w['nocc'] * 8 if is_df else 0)
    out = {
        'metric': 'J/K Fock-build wall-s/iter', 'value': ms_per_step * 1e-3, 'unit': 's',
        'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_per_step,
        'higher_is_better': False, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': args.workload, 'molecule': w['geom'], 'basis': w['basis'], 'nao': nao, 'path': path,
                   'direct_scf_tol': 1e-13, 'dm': 'SCF-like 2*C_occ*C_occ^T, orthonormal random C_occ, seed 1',
                   'l2_flush': '256 MiB memset between steps, outside the per-step CUDA-event pairs',
                   'parallelism': ('one build sharded over %d GPUs + 1 NCCL all-reduce of [J;K]' % world) if world > 1 else 'single GPU'},
        'e2e': {'value': e2e_ms_mean * 1e-3, 'unit': 's', 'h2d_bytes_per_step': int(h2d * (2 if omega2 else 1)),
                'd2h_bytes_per_step': int(nout * nao * nao * 8),
                'api': ('pyscf_b200.parallel.ShardedJK.get_jk' if world > 1 else
                        ('pyscf_b200.df.DF.get_jk' if is_df else 'pyscf_b200.jk.VHFOpt.get_jk')) + ' (pinned host dm)'},
        'gpu_launches': int(launches), 'setup_s': setup_s, 'clocks': clocks, 'roofline': roof,
        'wall_s_timed_region': t_wall,
        'device_vs_public_max_abs': float(dev_vs_pub),
        'parity': par,
    }
    if rank_ms is not None:   # residual limiter of the scaling: per-rank kernel time (min / max) vs the step
        out['per_rank_kernel_ms'] = {'min': min(rank_ms), 'max': max(rank_ms), 'all': rank_ms,
                                     'collective_and_sync_ms': ms_per_step - max(rank_ms)}
    if is_df:
        out['config']['naux'] = naux
        if naux2:
            out['config']['naux_long_range'] = naux2
        out['config']['nocc'] = w['nocc']
    else:
        out['quartets_computed'] = h.stats()['quartets_computed']
        out['quartets_screened'] = h.stats()['quartets_screened']
    if cpu is not None:
        out['cpu_baseline'] = cpu
    for hh in handles:
        hh.close()
    return out


# ------------------------------------------------------------------------------------------------------------------
def child_env(rank, world, port):
    env = dict(os.environ)
    env.update({'RANK': str(rank), 'LOCAL_RANK': os.environ.get('LOCAL_RANK', str(rank)), 'WORLD_SIZE': str(world),
                'MASTER_ADDR': '127.0.0.1', 'MASTER_PORT': str(port)})
    for k in list(env):     # the child builds its own rendezvous; drop the parent agent's elastic settings
        if k.startswith('TORCHELASTIC_') or k in ('GROUP_RANK', 'ROLE_RANK', 'ROLE_NAME', 'GROUP_WORLD_SIZE', 'ROLE_WORLD_SIZE'):
            env.pop(k)
    env['OMP_NUM_THREADS'] = str(host_threads())
    return env


def run_extra(name, steps, warmup, timeout, rank, world, base_port, idx, no_cpu, dump_dir):
    """Run one DF record in a child process of this rank; rank 0 returns the record (or an error record)."""
    tag = '%d_%d' % (base_port, idx)
    outp = '/tmp/b200jk_bench_%s.json' % tag
    failp = '/tmp/b200jk_bench_%s.fail' % tag
    if rank == 0:
        for p in (outp, failp):
            try:
                os.remove(p)
            except OSError:
                pass
    port = 20000 + (base_port + 101 * (idx + 1)) % 20000
    cmd = [sys.executable, os.path.abspath(__file__), '--child', '--workload', name, '--steps', str(steps), '--warmup', str(warmup),
           '--gpus', str(world), '--out', outp]
    if no_cpu:
        cmd.append('--no-cpu')
    if dump_dir:
        cmd += ['--dump-outputs', os.path.abspath(dump_dir)]
    t0 = time.time()
    log = open('/tmp/b200jk_bench_%s_r%d.log' % (tag, rank), 'w')
    proc = subprocess.Popen(cmd, env=child_env(rank, world, port), stdout=log, stderr=subprocess.STDOUT)
    status = 'ok'
    while True:
        rc = proc.poll()
        if rc is not None:
            if rc != 0:
                status = 'child exit code %d' % rc
                open(failp, 'w').write(status)
            break
        if os.path.exists(failp):
            status = 'another rank failed'
            proc.kill()
            break
        if time.time() - t0 > timeout:
            status = 'timeout after %d s' % timeout
            open(failp, 'w').write(status)
            proc.kill()
            break
        time.sleep(0.5)
    try:
        proc.wait(timeout=30)
    except Exception:
        pass
    log.close()
    if rank != 0:
        return None
    rec = None
    if os.path.exists(outp):
        try:
            rec = json.load(open(outp))
        except Exception as e:
            status = 'unreadable child record: %r' % e
    if rec is None:
        tail = ''
        try:
            tail = open('/tmp/b200jk_bench_%s_r0.log' % tag).read()[-600:]
        except Exception:
            pass
        rec = {'workload': name, 'error': status, 'log_tail': tail}
    rec['child_wall_s'] = time.time() - t0
    return rec


def run_ours(args, rank, world):
    import torch
    local = int(os.environ.get('LOCAL_RANK', rank))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    out = measure(args, rank, world, dist)
    if args.child:
        if rank == 0:
            json.dump(out, open(args.out, 'w'))
            print(json.dumps(out))
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    torch.cuda.empty_cache()
    # ---- the density-fitting configurations of BASELINE.json, one child process per rank each
    if not args.no_df and WORKLOADS[args.workload]['kind'] == 'direct':
        base_port = int(os.environ.get('MASTER_PORT', '29500'))
        df = {}
        t_start = time.time()
        for idx, (name, nmin, timeout) in enumerate(DF_EXTRAS):
            if world < nmin:
                if rank == 0:
                    df[name] = {'skipped': 'needs >= %d GPUs: %.1f GB of tensors (+ workspaces) against 180 GB of HBM per B200'
                                           % (nmin, TENSOR_GB[name])}
                continue
            left = args.df_budget - (time.time() - t_start)
            if world > 1:   # every rank takes the same decision
                tl = torch.tensor([left], device='cuda', dtype=torch.float64)
                dist.all_reduce(tl, op=dist.ReduceOp.MIN)
                left = float(tl[0])
            if left < 60:
                if rank == 0:
                    df[name] = {'skipped': 'time budget of the bench run exhausted (--df-budget %d s)' % args.df_budget}
                continue
            rec = run_extra(name, args.steps, args.warmup, min(timeout, left), rank, world, base_port, idx, args.no_cpu,
                            args.dump_outputs)
            if world > 1:
                dist.barrier()
            if rank == 0:
                df[name] = rec
        if rank == 0:
            out['df'] = df
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------------------------
def cpu_baseline_df(mol, dm, c_occ, workload):
    """Reference DF J/K algebra (df_jk.get_jk, pyscf/df/df_jk.py:362-380: dsymm-like half transform + dgemm) in numpy/OpenBLAS
    on a bounded sample of auxiliary rows of a random surrogate tensor of the right shape (timing only), scaled to naux."""
    from pyscf_b200.gto.mole import make_auxmol
    ncores = host_threads()
    try:
        from threadpoolctl import threadpool_limits
        ctx = threadpool_limits(limits=ncores)
    except Exception:
        ctx = None
    aux = make_auxmol(mol)
    naux, nao = aux.nao, mol.nao
    rows = max(8, min(naux, int(1e9 / (nao * nao * 8))))   # <= 1 GB sample
    rng = np.random.RandomState(0)
    eri1 = rng.standard_normal((rows, nao, nao))
    orbo = np.asfortranarray(c_occ * np.sqrt(2.0))
    dmtril = rng.standard_normal(nao * (nao + 1) // 2)
    packed = rng.standard_normal((rows, nao * (nao + 1) // 2))
    best = None
    for _ in range(2):
        t = time.perf_counter()
        vj = dmtril.dot(packed.T).dot(packed)
        buf = eri1.reshape(-1, nao).dot(orbo).reshape(rows, nao, -1)   # (P, nao, nocc): one threaded GEMM (the dsymm half transform)
        buf = np.ascontiguousarray(buf.transpose(0, 2, 1)).reshape(-1, nao)
        vk = buf.T.dot(buf)
        dt = (time.perf_counter() - t) * naux / rows
        best = dt if best is None else min(best, dt)
    nthr = None
    try:
        from threadpoolctl import threadpool_info
        nthr = max(i.get('num_threads', 0) for i in threadpool_info())
    except Exception:
        pass
    if ctx is not None:
        ctx.restore_original_limits()
    return {'value': best, 'unit': 's', 'cores': ncores, 'blas_threads': nthr, 'kind': 'port',
            'sample': '%d of %d auxiliary rows of %s (reference algebra df_jk.py:362-380 on a random tensor of the same shape: '
                      'two GEMV for J, batched matmul + GEMM for K, numpy/OpenBLAS), best of 2, time scaled by naux/rows'
                      % (rows, naux, workload), 'cpu_model': cpu_model()}


_LOOP_S = {}


def cpu_baseline(mol, dm, workload, keep=True, stride=1):
    """4-center CPU arm: the reference's own CVHFnr_direct_drv + nrs8 digestion + CVHFnrs8_prescreen compiled from the
    reference sources (oracle/_ref, kind "reference") when present, else the oracle's restatement (kind "port").
    Either way the integral function is oracle_cint.c's int2e_sph — libcint is not vendored in the reference tree.
    stride m > 1: a bounded sample.  The integral function handed to the driver evaluates only every m-th surviving shell
    quartet of each thread (the others return 0 and are skipped by the driver like vanishing libcint blocks), so
        T(m) = T_loop + W / m      (T_loop: quartet loop + prescreen over ALL quartets, W: integrals + digestion of the evaluated ones)
    and the full build is estimated as T_loop + m (T(m) - T_loop) with T_loop measured once by a run that evaluates nothing."""
    from oracle import oracle as O
    from oracle import ref_driver as R
    ncores = host_threads()
    nthr = R.set_threads(ncores)          # omp_set_num_threads + omp_get_max_threads: the count actually used
    info = {}
    t = time.perf_counter()
    if R.available():
        if stride > 1 and workload not in _LOOP_S:
            li = {}
            R.get_jk(mol, dm, hermi=1, sample_stride=1 << 30, info=li)
            _LOOP_S[workload] = li['driver_s']
        vj, vk = R.get_jk(mol, dm, hermi=1, sample_stride=max(1, stride), info=info)
        kind = 'reference'
        what = ('reference driver/screening/digestion (pyscf/lib/vhf/nr_direct.c, nr_direct_dot.c, optimizer.c compiled in '
                'place) + oracle McMurchie-Davidson int2e_sph (libcint absent)')
    else:
        stride = 1
        vj, vk, nq = O.get_jk(mol, dm, return_count=True)
        kind = 'port'
        what = 'oracle McMurchie-Davidson integrals + s8 digestion restatement, OpenMP over shell pairs'
    dt = time.perf_counter() - t
    t_loop = None
    if info.get('driver_s') is not None:
        # one SCF iteration = dm_cond + the driver; q_cond is per geometry (init_direct_scf, pyscf/scf/_vhf.py:151-206) like our setup_s
        dt = info['driver_s']
        if stride > 1:
            t_loop = min(_LOOP_S[workload], dt)
            dt_iter = info.get('dm_cond_s', 0.0) + t_loop + stride * (dt - t_loop)
        else:
            dt_iter = info.get('dm_cond_s', 0.0) + dt
    else:
        dt_iter = dt
    out = {'value': dt_iter, 'unit': 's', 'cores': ncores, 'omp_threads_used': nthr, 'kind': kind,
           'sample': ('one full J/K build of %s (every screened shell quartet), %s' % (workload, what)) if stride == 1 else
                     ('every %d-th surviving shell quartet of each OpenMP thread of one J/K build of %s (%d of %d quartets evaluated): driver '
                      '%.3f s, of which quartet loop + prescreen over all quartets %.3f s (measured by a run that evaluates nothing); full build '
                      'estimated as loop + %d x (driver - loop); %s'
                      % (stride, workload, info.get('evaluated', 0), info.get('calls', 0), dt, t_loop, stride, what)),
           'cpu_model': cpu_model()}
    if info.get('intor_thread_s') is not None and nthr and dt_iter > 0:
        f = min(1.0, info['intor_thread_s'] * stride / nthr / dt_iter)
        out['split'] = {'inside_integral_function_frac': f, 'driver_screening_digestion_frac': 1.0 - f,
                        'note': 'thread-seconds inside the oracle McMurchie-Davidson int2e_sph (x stride) / (threads x estimated build) vs the '
                                'reference C around it.  NON-LIBCINT INTEGRALS: libcint is several times faster per integral than this oracle, '
                                "and BASELINE.md's published whole-SCF time implies <~ 0.5 s per build for real PySCF on a modern host, so a "
                                'ratio against this arm overstates the speed-up over real PySCF'}
    if keep and stride == 1:
        out['vj'], out['vk'] = vj, vk
    return out


def run_reference(args, rank, world):
    if rank != 0:
        return
    w = WORKLOADS[args.workload]
    mol = build_mol(w)
    dm = scf_like_dm(mol.nao, w['nocc'])
    times = []
    base = None
    stride = args.ref_stride
    for k in range(args.warmup + args.steps):
        if w['kind'] == 'df':
            rng = np.random.RandomState(1)
            c_occ, _ = np.linalg.qr(rng.standard_normal((mol.nao, w['nocc'])))
            base = cpu_baseline_df(mol, dm, c_occ, args.workload)
        else:
            base = cpu_baseline(mol, dm, args.workload, keep=False, stride=stride)
        if k >= args.warmup:
            times.append(base['value'])
    v = float(np.mean(times))
    base['value'] = v
    out = {'impl': 'reference', 'metric': 'J/K Fock-build wall-s/iter', 'value': v, 'unit': 's', 'n_gpus': world,
           'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': v * 1e3, 'higher_is_better': False,
           'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
           'config': {'workload': args.workload, 'molecule': w['geom'], 'basis': w['basis'], 'nao': mol.nao,
                      'path': ('DF J/K (reference algebra on the host)' if w['kind'] == 'df'
                               else '4-center direct J/K (hermi=1, with_j, with_k)'), 'direct_scf_tol': 1e-13,
                      'dm': 'SCF-like 2*C_occ*C_occ^T, orthonormal random C_occ, seed 1',
                      'parallelism': 'host cores of rank 0 (OpenMP), no GPU',
                      'note': 'reference CPU path: the reference driver/screening/digestion compiled from its own sources '
                              '(oracle/_ref) around the oracle integral function; libcint itself is not vendored in the '
                              'reference tree (DESIGN.md section 2): NON-LIBCINT INTEGRALS, the ratio against this arm overstates '
                              'the speed-up over real PySCF (see cpu_baseline.split)'},
           'cpu_baseline': base,
           'e2e': {'value': v, 'unit': 's', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='benzene-ccpvtz-direct', choices=sorted(WORKLOADS))
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--no-df', action='store_true', help='headline workload only (no "df" records)')
    ap.add_argument('--df-budget', type=int, default=560, help='seconds the DF records of one run may take in total')
    ap.add_argument('--ref-stride', type=int, default=8, help='--impl reference: evaluate every m-th surviving shell quartet per step')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write J and K of the last timed step of every record as DIR/<workload>_<J|K|K_omega>.npy (float64)')
    ap.add_argument('--child', action='store_true', help=argparse.SUPPRESS)
    ap.add_argument('--out', default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    if args.impl == 'reference':
        run_reference(args, rank, world)
    else:
        if args.warmup < 3:
            args.warmup = 3
        run_ours(args, rank, world)


if __name__ == '__main__':
    main()
