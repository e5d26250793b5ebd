"""Which image sizes the FFT operators take (csrc/fft_plan.h), checked without a GPU: the size class and the plan of
the mixed-radix path, the refusal message of the other sizes, and that a supported size on a host without a device
fails with SBD_E_NODEVICE (there is no CPU fallback)."""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "semi-blind-image-deblurring-problems-with-tv_b200", "csrc")

PROBE = r"""
#include "fft_plan.h"
#include <cstdio>
#include <cstdlib>
int main(int argc, char** argv) {
    for (int i = 1; i + 1 < argc; i += 2) {
        const int r = atoi(argv[i]), c = atoi(argv[i + 1]);
        printf("%d %d|%s\n", r, c, sbd::fft_size_error(r, c).c_str());
    }
    for (int n = 2; n <= 4096; ++n) {
        sbd::AnyPlan p;
        if (!sbd::any_plan(n, &p)) continue;
        long prod = 1;
        printf("plan %d %d %d", n, p.nst, p.T);
        for (int s = 0; s < p.nst; ++s) { printf(" %d", p.r[s]); prod *= p.r[s]; }
        printf(" = %ld\n", prod);
    }
    return 0;
}
"""

SIZES = [(481, 512), (512, 4097), (480, 640), (2160, 3840), (7, 9), (512, 512), (512, 962), (4096, 4096), (4097, 4096)]


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    d = tmp_path_factory.mktemp("plan")
    src = d / "probe.cpp"
    src.write_text(PROBE)
    exe = d / "probe"
    subprocess.run(["g++", "-std=c++17", "-I", CSRC, "-o", str(exe), str(src)], check=True)
    args = [str(v) for s in SIZES for v in s]
    out = subprocess.run([str(exe)] + args, capture_output=True, text=True, check=True).stdout.splitlines()
    msgs = {}
    plans = {}
    for ln in out:
        if ln.startswith("plan "):
            f = ln.split()
            plans[int(f[1])] = (int(f[2]), int(f[3]), [int(v) for v in f[4:-2]], int(f[-1]))
        else:
            k, m = ln.split("|", 1)
            msgs[tuple(map(int, k.split()))] = m
    return msgs, plans


def smooth(n):
    for f in (2, 3, 5, 7):
        while n % f == 0:
            n //= f
    return n == 1


def test_refusals_name_the_side_and_factor(probe):
    msgs, _ = probe
    assert msgs[(481, 512)] == "rows = 481 = 13·37: FFT lengths need prime factors ≤ 7"
    assert msgs[(512, 4097)].startswith("cols = 4097 = 17·241") and "4096" in msgs[(512, 4097)]
    assert msgs[(4097, 4096)].startswith("rows = 4097")
    assert "cols = 962 = 2·13·37" in msgs[(512, 962)]
    for ok in [(480, 640), (2160, 3840), (7, 9), (512, 512), (4096, 4096)]:
        assert msgs[ok] == "", ok


def test_plans_cover_every_smooth_length(probe):
    _, plans = probe
    assert set(plans) == {n for n in range(2, 4097) if smooth(n)}
    for n, (nst, T, radices, prod) in plans.items():
        assert prod == n and nst == len(radices) and nst <= 7
        assert set(radices) <= {2, 3, 4, 5, 7, 8}
        assert T % 32 == 0 and T <= 512
        # a thread owns at most 16 complex values per stage
        for R in radices:
            assert (16 // R) * T * R >= n


def test_supported_sizes_have_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the -m gpu tests")
    import sys
    sys.path.insert(0, ROOT)
    import sbd_b200
    from sbd_b200 import SbdError
    for shape in [(480, 640), (243, 375)]:
        with pytest.raises(SbdError) as e:
            sbd_b200.Engine(shape[0], shape[1])
        assert e.value.code == -3, e.value.msg
