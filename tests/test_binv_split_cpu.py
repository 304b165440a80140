"""The inversion sampler in two parts (include/mmq_sampler.h: mmq_binv_setup once per draw, mmq_binv_attempt per
attempt, which k_alloc_chain runs apart) against the single sequential loop it was split from, written out here: the
same integers over a grid of (n, p) on both sides of p = 1/2 and up to the BTRS boundary n p = 10.  CPU only: the
header is compiled by the host compiler with contraction off, as for the CPU replay."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SRC = r"""
#include "mmq_sampler.h"
/* BINV as one loop: the setup inline, the attempts one after the other */
static int64_t binv_loop(const mmq_rng* g, uint32_t block0, int64_t n, double p) {
  const double dn = (double)n;
  const double q = 1.0 - p;
  const double s = p / q;
  const double a = (dn + 1.0) * s;
  const double r0 = mmq_exp(dn * mmq_log1p(-p));
  for (uint32_t att = 0;; ++att) {
    uint32_t w[4];
    mmq_rng_block(g, block0 + att, w);
    double r = r0;
    double u = mmq_uniform52(w[0], w[1]);
    int64_t x = 0;
    while (u > r) {
      u -= r;
      x += 1;
      if (x > n) break;
      r *= (a * mmq_inv_small(x) - s);
    }
    if (x <= n) return x;
  }
}
/* out[2 i] = the loop, out[2 i + 1] = mmq_binomial (setup + attempts) for draws i = 0 .. cnt-1 of class ids id0 + i */
extern "C" void draw_both(uint32_t seed, uint64_t id0, int64_t cnt, int64_t n, double p, int64_t* out) {
  for (int64_t i = 0; i < cnt; ++i) {
    mmq_rng g;
    mmq_rng_init(&g, seed, MMQ_STREAM_ALLOC, id0 + (uint64_t)i, 3u);
    const uint32_t b0 = MMQ_CHAIN_BLOCK(5);
    out[2 * i] = p > 0.5 ? n - binv_loop(&g, b0, n, 1.0 - p) : binv_loop(&g, b0, n, p);
    out[2 * i + 1] = mmq_binomial(&g, b0, n, p);
  }
}
"""


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    d = tmp_path_factory.mktemp("binv")
    src, so = d / "binv.cpp", d / "binv.so"
    src.write_text(SRC)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-I", os.path.join(ROOT, "include"),
                           "-o", str(so), str(src)])
    L = C.CDLL(str(so))
    L.draw_both.argtypes = [C.c_uint32, C.c_uint64, C.c_int64, C.c_int64, C.c_double, C.c_void_p]
    L.draw_both.restype = None
    return L


def _grid():
    for n in (2, 3, 7, 33, 100, 1000, 20000):
        for p in (1e-9, 1e-4, 0.003, 0.05, 0.2, 0.4999, 0.5, 0.5001, 0.8, 0.97, 1 - 1e-6):
            if min(p, 1 - p) * n < 10:   # the inversion regime of mmq_binomial
                yield n, p


@pytest.mark.parametrize("n,p", list(_grid()))
def test_split_binv_equals_sequential_loop(lib, n, p):
    cnt = 4000
    out = np.zeros(2 * cnt, np.int64)
    lib.draw_both(20261022, (1 << 32) * 7 + n, cnt, n, p, out.ctypes.data)
    loop, split = out[0::2], out[1::2]
    assert np.array_equal(loop, split)
    assert loop.min() >= 0 and loop.max() <= n
