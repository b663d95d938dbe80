"""CPU: the C-ABI library loads, exports every symbol include/aoadmm.h declares, and the host-side mirror behaves
(no compute calls - there is no GPU here)."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    src = open(os.path.join(ROOT, 'include', 'aoadmm.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return sorted(set(re.findall(r'\b(aoadmm_[a-z0-9_]+)\s*\(', src)))


def test_library_exports_every_declared_symbol(ab):
    names = header_functions()
    assert 'aoadmm_run' in names and 'aoadmm_create' in names and len(names) >= 17
    for n in names:
        assert hasattr(ab._capi.lib, n), n
    assert sorted(ab._capi.EXPORTS) == names
    assert ab._capi.lib.aoadmm_abi_version() == 4


def test_struct_layouts_match_header(ab, tmp_path):
    """compile include/aoadmm.h with gcc and compare sizeof/offsetof with the ctypes mirror."""
    import subprocess
    c = ab._capi
    structs = {'aoadmm_constraint': c.Constraint, 'aoadmm_object': c.Object, 'aoadmm_problem': c.Problem,
               'aoadmm_dist': c.Dist, 'aoadmm_options': c.Options, 'aoadmm_out': c.Out}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "aoadmm.h"', 'int main(void){']
    for cname, cls in structs.items():
        lines.append('printf("%s %%zu\\n", sizeof(%s));' % (cname, cname))
        for fname, _ in cls._fields_:
            lines.append('printf("%s.%s %%zu\\n", offsetof(%s, %s));' % (cname, fname, cname, fname))
    lines.append('return 0;}')
    src = tmp_path / 'layout.c'
    src.write_text('\n'.join(lines))
    exe = tmp_path / 'layout'
    subprocess.check_call(['gcc', '-I', os.path.join(ROOT, 'include'), str(src), '-o', str(exe)])
    got = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).splitlines())
    for cname, cls in structs.items():
        assert int(got[cname]) == ctypes.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert int(got['%s.%s' % (cname, fname)]) == getattr(cls, fname).offset, (cname, fname)


def test_no_device_is_an_error_not_a_fallback(ab):
    if ab.device_count() > 0:
        pytest.skip('a GPU is present')
    X = np.zeros((4, 3, 2))
    U = [np.ones((s, 2)) for s in X.shape]
    with pytest.raises(ab.AoadmmError) as e:
        ab.mttkrp(X, U, 1)
    assert e.value.status_name == 'NO_DEVICE'
    with pytest.raises(ab.AoadmmError):
        ab.prox(('non-negativity',), np.zeros((3, 2)))


def test_invalid_arguments_rejected_without_device(ab):
    c = ab._capi
    assert c.lib.aoadmm_create(None, None, None) == 1
    h = c.HandleP()
    assert c.lib.aoadmm_create(None, None, ctypes.byref(h)) != 0
    assert b'NULL' in c.lib.aoadmm_last_error(None)
    assert c.lib.aoadmm_run(None, None, None) == 1
    assert c.lib.aoadmm_destroy(None) == 0
    # the one-caller multi-GPU form (ABI 4): same conventions
    assert c.lib.aoadmm_create_multi(None, 2, None, None) == 1
    assert c.lib.aoadmm_create_multi(None, 2, None, ctypes.byref(h)) != 0 and not h.value
    assert b'NULL' in c.lib.aoadmm_last_error(None)
    n = ctypes.c_int32(7)
    assert c.lib.aoadmm_gpu_count(None, ctypes.byref(n)) == 1
    assert c.lib.aoadmm_comm_release() == 0           # nothing cached: a no-op


def test_constraint_spec_mapping(ab):
    spec, _ = ab.constraint_spec(('box', -1.0, 2.0))
    assert (spec.kind, spec.p0, spec.p1) == (2, -1.0, 2.0)
    spec, _ = ab.constraint_spec(('unimodality', True))
    assert (spec.kind, spec.p0) == (7, 1.0)
    spec, _ = ab.constraint_spec(('TV regularization', 1e-3))
    assert (spec.kind, spec.p0) == (19, 1e-3)
    spec, keep = ab.constraint_spec(('quadratic regularization', 0.5, np.eye(3)))
    assert spec.kind == 17 and spec.matrix_n == 3 and keep is not None
    assert ab.constraint_spec(None)[0].kind == 0
    with pytest.raises(ValueError):
        ab.constraint_spec(('no such constraint',))
    # every named spec of constraints_to_prox.m:13-91 is known (the names, in the file's order, are stored in
    # tests/golden/constraints_to_prox_names.txt)
    with open(os.path.join(ROOT, 'tests', 'golden', 'constraints_to_prox_names.txt')) as f:
        ref = f.read().split('\n')[:-1]
    assert len(ref) == 21 and ref[-1] == 'custom'
    assert sorted(ab._capi.CONSTRAINT_KINDS) == sorted(ref)


def test_shard_range_partitions(ab):
    for extent in (1, 7, 256, 1000, 2048):
        for world in (1, 2, 3, 4, 8):
            parts = [ab.shard_range(extent, r, world) for r in range(world)]
            assert parts[0][0] == 0 and parts[-1][1] == extent
            assert all(parts[i][1] == parts[i + 1][0] for i in range(world - 1))
            sizes = [hi - lo for lo, hi in parts]
            assert max(sizes) - min(sizes) <= 1


def test_unsupported_inputs_raise_before_touching_the_device(ab):
    from oracle import problem_gen as pg
    Z, G, _ = pg.config_script6(seed=0, sz=(6, 7, 5, 6, 8, 7, 9))
    Zk = dict(Z, loss_function=['KL', 'Frobenius', 'Frobenius'])
    with pytest.raises(ab.AoadmmError) as e:
        ab.cmtf_fun_AOADMM(Zk, pg.znorm_const(Z), G, None, None, None, None, pg.default_options())
    assert e.value.status_name == 'UNSUPPORTED'
    Zm = dict(Z, miss=[np.ones((3, 3, 3)), None, None])       # cmtf:missingData:maskSizeMismatch (cmtf_AOADMM.m:85-88)
    with pytest.raises(ab.AoadmmError):
        ab.cmtf_fun_AOADMM(Zm, pg.znorm_const(Z), G, None, None, None, None, pg.default_options())
    Zt = dict(Z, constraints=[('tPARAFAC2', 0.1)] + list(Z['constraints'][1:]))              # cmtf_AOADMM.m:33-39
    with pytest.raises(ValueError):
        ab.cmtf_AOADMM(Zt, G, pg.default_options())
    Zp, Gp, _ = pg.config_single_par2(I=6, Jk=(5, 4), R=2, seed=0)
    for bad, msg in (([np.ones((6, 5))], 'cell array of length'),                              # :101-104
                     ([np.full((6, 5), 0.5), np.ones((6, 4))], 'logical or binary'),            # :107-114
                     ([np.ones((6, 5)), np.ones((6, 5))], 'size does not match')):              # :115-118
        with pytest.raises(ab.AoadmmError) as e:
            ab.cmtf_fun_AOADMM(dict(Zp, miss=[bad]), pg.znorm_const(Zp), Gp, None, None, None, None, pg.default_options())
        assert msg in str(e.value), (msg, str(e.value))


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, 'matlab-code_b200')
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h', '.cpp', '.m')):
                txt = open(os.path.join(dp, f), errors='replace').read()
                assert 'import oracle' not in txt and 'from oracle' not in txt, os.path.join(dp, f)


def test_mex_gateway_compiles_against_stub_mex_header():
    """MATLAB is not available offline: the gateway source is at least compiled (syntax + C-ABI signatures) against a
    declarations-only mex.h, and must bind only symbols that include/aoadmm.h declares."""
    import re
    import subprocess
    header = open(os.path.join(ROOT, 'include', 'aoadmm.h')).read()
    declared = set(re.findall(r'\b(aoadmm_[a-z_0-9]+)\s*\(', header))
    for name in ('aoadmm_mex.cpp', 'aoadmm_nvecs_mex.cpp'):
        src = os.path.join(ROOT, 'matlab-code_b200', 'matlab', name)
        subprocess.check_call(['g++', '-std=c++17', '-fsyntax-only', '-Wall', '-I', os.path.join(ROOT, 'tests', 'stubs'),
                               '-I', os.path.join(ROOT, 'include'), src])
        used = set(re.findall(r'\b(aoadmm_[a-z_0-9]+)\s*\(', open(src).read())) - {'aoadmm_mex', 'aoadmm_nvecs_mex'}
        assert used and used <= declared, used - declared
    nv = open(os.path.join(ROOT, 'matlab-code_b200', 'matlab', 'cmtf_nvecs.m')).read()
    assert nv.startswith('function U = cmtf_nvecs(Z,n,r)')
    shim = open(os.path.join(ROOT, 'matlab-code_b200', 'matlab', 'cmtf_fun_AOADMM.m')).read()
    assert shim.startswith('function [G,out] = cmtf_fun_AOADMM(Z,Znorm_const,G,fh,gh,lscalar,uscalar,options)')


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the engine) needs no GPU: one JSON line with the
    contract keys, the CPU baseline description and an end-to-end block without device copies."""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0'],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line['impl'] == 'reference' and line['metric'] == 'ao_admm_outer_iters_per_s' and line['unit'] == 'outer_iters/s'
    assert line['higher_is_better'] is True and line['n_gpus'] == 1 and line['steps'] == 1 and line['dtype'] == 'f64'
    assert line['value'] > 0 and line['ms_per_step'] > 0 and line['vs_baseline'] is None and line['data'] == 'synthetic'
    assert 'workload' in line['config'] and 'model' not in line['config']
    cb = line['cpu_baseline']
    assert cb['kind'] in ('port', 'reference') and cb['cores'] >= 1 and cb['sample'] and cb['value'] == line['value']
    e2e = line['e2e']
    assert e2e['value'] == line['value'] and e2e['h2d_bytes_per_step'] == 0 and e2e['d2h_bytes_per_step'] == 0


def test_init_front_end_host_logic_matches_oracle_without_device(ab):
    """ab.init_coupled_AOADMM_CMTF (init_coupled_AOADMM_CMTF.m:37-169) with random factors and no constrained mode is
    pure host logic: same shapes and, with the same random stream, the same numbers as the oracle's restatement, for
    every coupling type and for PARAFAC2 objects."""
    from oracle import problem_gen as pg
    cases = [pg.config_linear_coupling(ct, seed=ct, constrained=False)[0] for ct in (1, 2, 3, 4)]
    cases.append(pg.config_single_par2(seed=1, constrained=(0, 0, 0))[0])
    Zs, _, _ = pg.config_script6(seed=1, sz=(6, 7, 5, 6, 8, 7, 9))
    cases.append(dict(Zs, constrained_modes=[0] * 7))
    for Z in cases:
        P = len(Z['modes'])
        R = 3
        lambdas = []
        for p in range(P):
            lambdas.append([1.0] * (4 if (Z['coupling'].get('coupling_type') in ([2], [4]) and p == 0) else R))
        r1, r2 = np.random.RandomState(5), np.random.RandomState(5)
        io = {'lambdas_init': lambdas, 'nvecs': 0, 'normalize': 1}
        Go = pg.init_coupled_AOADMM_CMTF(Z, dict(io, distr=[pg.d_rand] * len(Z['size'])), r2)
        Gd = ab.init_coupled_AOADMM_CMTF(Z, dict(io, distr=[lambda a, b: r1.rand(a, b)] * len(Z['size'])), rng=r1)
        for key in ('fac', 'coupling_fac', 'coupling_dual_fac', 'P', 'DeltaB', 'mu_DeltaB'):
            for a, b in zip(Gd[key], Go[key]):
                if b is None:
                    assert a is None
                elif isinstance(b, list):
                    assert len(a) == len(b) and all(np.array_equal(x, y) for x, y in zip(a, b)), key
                else:
                    assert np.array_equal(a, b), key


def test_every_entry_point_is_documented_in_integration_md():
    """INTEGRATION.md maps every C-ABI entry point to the reference interface it replaces."""
    import re
    header = open(os.path.join(ROOT, 'include', 'aoadmm.h')).read()
    doc = open(os.path.join(ROOT, 'INTEGRATION.md')).read()
    funcs = set(re.findall(r'\b(aoadmm_[a-z_0-9]+)\s*\(', header))
    funcs -= {'aoadmm_status', 'aoadmm_abi_version', 'aoadmm_device_count'}   # the status enum; two trivial queries
    missing = sorted(f for f in funcs if f not in doc)
    assert not missing, missing
