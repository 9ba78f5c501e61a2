"""Launch plan of the objective (nmrfit_b200/csrc/objective_plan.h) compiled for the host: one case per branch - which
kernel runs, with what geometry and scratch, and each refusal.  The expected values are the choices the library made
before the plan was one function (tools/objective_plan_equiv.cpp compares the two over the whole grid)."""
import ctypes
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FP64, FP32 = 0, 1
AUTO, GENERAL, UNIFORM = 0, 1, 2
KERNELS = ('general', 'uniform', 'stream', 'f32_uniform', 'f32_general')
FIELDS = ('kernel', 'threads', 'r', 'tb', 'sp', 'variant', 'stages', 'occ', 'sub', 'n_tiles', 'nw', 'nsum', 'tile_major',
          'gpc', 'prep_g', 'prep_threads', 'smem', 'prep_smem', 'part_per', 'far', 'mask', 'refuse')

SRC = r'''
#include "%s/nmrfit_b200/csrc/objective_plan.h"
#include <cstring>
extern "C" void plan(int N, int P, int S, int B, int precision, int fit_im, int uniform, int algorithm, int threads,
                     int r, int tb, int sp, int far_cells, long long* out, char* why) {
    const nmrfit::ObjTune user{threads, r, tb, sp, -1, 0, 0};
    const nmrfit::ObjPlan p = nmrfit::objective_plan(N, P, S, B, precision, fit_im, uniform != 0, algorithm, user, far_cells);
    const long long v[] = {p.kernel, p.t.threads, p.t.r, p.t.tb, p.t.sp, p.t.variant, p.t.stages, p.t.occ, p.sub,
                           p.n_tiles, p.nw, p.nsum, p.tile_major, p.gpc, p.prep_g, p.prep_threads, (long long)p.smem,
                           (long long)p.prep_smem, (long long)p.part_per, (long long)p.far, (long long)p.mask, p.refuse};
    std::memcpy(out, v, sizeof v);
    std::strcpy(why, p.why ? p.why : "");
}
'''


@pytest.fixture(scope='module')
def lib(tmp_path_factory):
    d = tmp_path_factory.mktemp('plan')
    src, so = d / 'plan.cpp', str(d / 'plan.so')
    src.write_text(SRC % ROOT)
    subprocess.run(['g++', '-O2', '-std=c++17', '-Wall', '-Werror', '-shared', '-fPIC', '-o', so, str(src)], check=True)
    return ctypes.CDLL(so)


def plan(lib, N, P, S, B=1, precision=FP64, fit_im=0, uniform=True, algorithm=AUTO, threads=0, r=0, tb=0, sp=0,
         far_cells=0):
    out = (ctypes.c_longlong * len(FIELDS))()
    why = ctypes.create_string_buffer(256)
    lib.plan(N, P, S, B, precision, fit_im, int(uniform), algorithm, threads, r, tb, sp, far_cells, out, why)
    p = dict(zip(FIELDS, out))
    p['kernel'] = KERNELS[p['kernel']]
    p['why'] = why.value.decode()
    return p


def check(p, **want):
    assert {k: p[k] for k in want} == want


def test_headline_shape_streams(lib):
    # 6 peaks x 4,096 points x 65,536 particles: two stages of 8 particles, two CTAs per SM, four far-field cells
    p = plan(lib, 4096, 6, 65536)
    check(p, kernel='stream', threads=256, r=8, tb=6, sp=8, variant=1, stages=2, occ=2, sub=4, n_tiles=2, nw=8,
          nsum=1, tile_major=1, gpc=7, prep_g=16, prep_threads=256, smem=114720, prep_smem=12032, part_per=32, far=640,
          mask=160, refuse=0)


def test_single_fit_runs_one_group_per_cta(lib):
    p = plan(lib, 4096, 6, 204)
    check(p, kernel='uniform', threads=256, r=8, sp=1, variant=0, sub=4, n_tiles=2, nw=1, tile_major=0, prep_g=1,
          prep_threads=128, smem=53680, prep_smem=752, part_per=4)


def test_other_exp_table_runs_one_group_per_cta(lib):
    # the streamed kernel is built for the default table only
    p = plan(lib, 4096, 6, 65536, tb=8)
    check(p, kernel='uniform', threads=256, r=8, tb=8, sp=6, variant=0, sub=4, nw=1, prep_g=16, smem=75216)


def test_fit_im(lib):
    # the sum over peaks runs the general kernel; the reference's fit_im stays on the uniform axis, with two sums
    check(plan(lib, 4096, 6, 65536, fit_im=2), kernel='general', threads=128, r=4, sp=16, sub=1, n_tiles=8, nw=1,
          nsum=2, prep_threads=0, smem=20096, part_per=16)
    check(plan(lib, 4096, 6, 65536, fit_im=1), kernel='stream', nsum=2, smem=114720)


def test_fp32_uniform_runs_r8_when_asked_for_16(lib):
    # the particle tile is still chosen for 16 points per thread, then the kernel runs 8
    p = plan(lib, 4096, 6, 1000, precision=FP32, r=16)
    check(p, kernel='f32_uniform', threads=256, r=8, sp=1, sub=1, n_tiles=2, nw=1, tile_major=0, prep_g=3,
          prep_threads=256, smem=51504, prep_smem=2256, part_per=4, far=160, mask=32)


def test_fp32_non_uniform_axis_runs_256_by_4(lib):
    p = plan(lib, 4096, 6, 1000, precision=FP32, uniform=False)
    check(p, kernel='f32_general', threads=256, r=4, sp=13, n_tiles=4, nsum=1, prep_threads=0, smem=2704, part_per=16)
    check(plan(lib, 1500, 6, 12, precision=FP32, uniform=False), kernel='f32_general', threads=256, r=4, sp=1,
          n_tiles=2, smem=208, part_per=6)


@pytest.mark.parametrize('kw,code,msg', [
    (dict(r=2), -1, 'points_per_thread must be 4, 8 or 16 for the uniform-axis kernel'),
    (dict(r=16, uniform=False), -1, 'points_per_thread must be 2, 4 or 8 for the general kernel'),
    (dict(algorithm=UNIFORM, uniform=False), -3,
     'the uniform-axis kernel needs uniformly spaced w in every spectrum and fit_im off'),
    (dict(precision=FP32, fit_im=1), -1,
     'fit_im is not available in FP32 mode (the Kramers-Kronig term runs in FP64 only)'),
])
def test_refusals(lib, kw, code, msg):
    p = plan(lib, 4096, 6, 100, **kw)
    assert (p['refuse'], p['why']) == (code, msg)


def test_refusal_order(lib):
    # the uniform-axis refusal comes before the FP32 fit_im one, which comes before points_per_thread
    p = plan(lib, 4096, 6, 100, precision=FP32, fit_im=2, algorithm=UNIFORM, r=16)
    assert p['refuse'] == -3
    p = plan(lib, 4096, 6, 100, precision=FP32, fit_im=1, uniform=False, r=16)
    assert p['why'].startswith('fit_im is not available')
