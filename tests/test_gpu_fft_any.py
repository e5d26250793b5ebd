"""GPU parity of the mixed-radix FFT path (fft_any.cuh): image sizes that are not powers of two, every side in
[2, 4096] with prime factors <= 7.  Operators against the numpy oracle (relative error 1e-12, per image of a batch),
large shapes against cuFFT, the likelihood closures, the setup stage, SALSA, SAPG against the oracle fed the same
noise (1e-6), sharding, and the Python / MATLAB surfaces."""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from conftest import rel, ROOT

pytestmark = pytest.mark.gpu

TOL = 1e-12
TRAJ_TOL = 1e-6
PSI = {0: (0.4, 0.3), 1: (0.4, 3.5), 2: (0.3,)}

SHAPES = [(480, 640), (600, 800), (243, 375), (343, 125), (375, 512), (512, 375), (512, 768), (49, 343), (20, 28)]


@pytest.fixture(scope="module")
def sbd():
    import sbd_b200
    return sbd_b200


@pytest.fixture(scope="module")
def O():
    import oracle
    import scipy.fft
    w = os.cpu_count() or 1
    oracle.operators.set_fft(lambda a: scipy.fft.fft2(a, workers=w), lambda a: scipy.fft.ifft2(a, workers=w))
    yield oracle
    oracle.operators.set_fft(np.fft.fft2, np.fft.ifft2)


class NoiseTape:
    def __init__(self, seed):
        self.rng = np.random.default_rng(seed)
        self.tape = []
        self.record = False

    def __call__(self, shape):
        z = self.rng.standard_normal(shape)
        if self.record:
            self.tape.append(z)
        return z


def _crop(img, shape):
    """a natural image of any shape: the fixture tiled (mirrored) and cropped"""
    reps = (-(-shape[0] // img.shape[0]) + 1, -(-shape[1] // img.shape[1]) + 1)
    t = np.block([[img if (i + j) % 2 == 0 else img[::-1, ::-1] for j in range(reps[1])] for i in range(reps[0])])
    return np.ascontiguousarray(t[:shape[0], :shape[1]])


# ---------------------------------------------------------------- operators
@pytest.mark.parametrize("model", [0, 1, 2])
@pytest.mark.parametrize("shape,psf_size", [(s, 7) for s in SHAPES] + [((7, 9), 7)])
def test_operators_vs_oracle(sbd, O, model, shape, psf_size):
    B = 3
    rng = np.random.default_rng(shape[0] * 31 + shape[1] + model)
    x = rng.uniform(0, 255, (B,) + shape)
    eng = sbd.Engine(shape[0], shape[1], psf_size, model, 0.0, max_batch=B)
    cl = O.operators.closures(model, shape, psf_size, 0.0)
    psi = PSI[model]
    ops = [(0, cl["A"]), (1, cl["AT"])] + [(2 + i, d) for i, d in enumerate(cl["dif"])]
    for op, f in ops:
        got = eng.blur(x, psi, op)
        for b in range(B):
            assert rel(got[b], f(x[b], *psi)) < TOL, (shape, model, op, b)
    nk = 2 if model == 2 else 3
    for which in range(nk):
        want = O.psf.resize(O.psf.taps(model, psf_size, psi, 0.0, which), shape)
        assert rel(eng.psf_spectrum(psi, which), want) < TOL, (shape, model, which)
    eng.close()


def test_unsupported_sizes_name_the_factor(sbd):
    """Sizes with a prime factor above 7 keep SBD_E_UNSUPPORTED for the FFT operators, with the factor in the message;
    the TV entry points still take them."""
    from sbd_b200 import SbdError
    eng = sbd.Engine(481, 512, 7, 0, 0.0)
    x = np.random.default_rng(0).uniform(0, 1, (481, 512))
    with pytest.raises(SbdError) as e:
        eng.blur(x, PSI[0], 0)
    assert e.value.code == -6 and "481" in e.value.msg and "13" in e.value.msg, e.value.msg
    assert np.isfinite(eng.tvnorm(x))
    eng.close()


def test_live_engines_of_different_sizes_alternate(sbd):
    """The shared-memory opt-in of the mixed-radix kernels belongs to the device, not to a context: a second live
    context with shorter lines (3200 vs 4000 rows) must not break the next call on the first one."""
    rng = np.random.default_rng(8)
    e1 = sbd.Engine(4000, 3000, 7, 0, 0.0)
    e2 = sbd.Engine(3200, 2400, 7, 0, 0.0)
    x1 = rng.uniform(0, 255, (4000, 3000))
    x2 = rng.uniform(0, 255, (3200, 2400))
    a1 = e1.blur(x1, PSI[0], 0)
    a2 = e2.blur(x2, PSI[0], 0)
    assert np.array_equal(e1.blur(x1, PSI[0], 0), a1)
    assert np.array_equal(e2.blur(x2, PSI[0], 1), e2.blur(x2, PSI[0], 1))
    assert np.array_equal(e1.blur(x1, PSI[0], 0), a1)
    assert np.array_equal(e2.blur(x2, PSI[0], 0), a2)
    e1.close()
    e2.close()


# ---------------------------------------------------------------- cuFFT at large shapes
def _cufft_blur(x, taps, conj=False):
    import torch
    b, n0, n1 = x.shape
    pad = torch.zeros((n0, n1), dtype=torch.float64, device=x.device)
    t = taps.shape[0]
    pad[:t, :t] = torch.from_numpy(np.ascontiguousarray(taps)).to(x.device)
    H = torch.fft.rfft2(pad)
    if conj:
        H = torch.conj(H)
    return torch.fft.irfft2(torch.fft.rfft2(x) * H, s=(n0, n1))


@pytest.mark.parametrize("shape", [(2160, 3840), (3000, 4000)])
@pytest.mark.parametrize("model", [0, 1, 2])
def test_large_vs_cufft(sbd, O, shape, model):
    import torch
    from sbd_b200._lib import lib, c_double_p
    B = 4
    rows, cols = shape
    eng = sbd.Engine(rows, cols, 7, model, 0.0, max_batch=B)
    g = torch.Generator(device="cuda").manual_seed(rows + model)
    x_t = torch.rand((B, cols, rows), dtype=torch.float64, device="cuda", generator=g) * 255.0    # [b][col][row]
    out = torch.empty_like(x_t)
    psi = np.zeros(2); psi[:len(PSI[model])] = PSI[model]
    for op in range(3 if model == 2 else 4):
        which = {0: 0, 1: 0, 2: 1, 3: 2}[op]
        taps = O.psf.taps(model, 7, PSI[model], 0.0, which)
        want = _cufft_blur(x_t, taps.T, conj=(op == 1))
        rc = lib.sbd_blur_dev(eng._h, x_t.data_ptr(), psi.ctypes.data_as(c_double_p), op, out.data_ptr(), B)
        assert rc == 0, lib.sbd_last_error(eng._h)
        lib.sbd_synchronize(eng._h)
        for b in range(B):
            r = (torch.linalg.vector_norm(out[b] - want[b]) / torch.linalg.vector_norm(want[b])).item()
            assert r < TOL, (shape, model, op, b, r)
    eng.close()


# ---------------------------------------------------------------- likelihood, setup stage, SALSA
@pytest.mark.parametrize("shape", [(243, 375), (480, 640)])
@pytest.mark.parametrize("model", [0, 1, 2])
def test_likelihood(sbd, O, cman, shape, model):
    rng = np.random.default_rng(model + shape[0])
    xc = _crop(cman, shape)
    cl = O.operators.closures(model, shape, 7, 0.0)
    y = cl["A"](xc, *PSI[model]) + 2.0 * rng.standard_normal(shape)
    x = np.abs(xc + 3.0 * rng.standard_normal(shape))
    psi = {0: (0.5, 0.35), 1: (0.8, 6.0), 2: (0.15,)}[model]
    s2, th = 7.5, 0.04
    f, gradF, grads, gsig = O.operators.likelihood_closures(cl, y, x.size)
    eng = sbd.engine_for(shape, 7, model, 0.0)
    got = eng.likelihood(x, y, psi, s2, th)
    args = (*psi, s2)
    assert abs(got["f"] - f(x, *args)) <= TOL * abs(f(x, *args))
    assert rel(got["gradF"], gradF(x, *args)) < TOL
    for i, gr in enumerate(grads):
        scale = np.sum(np.abs(cl["dif"][i](x, *psi) * (cl["A"](x, *psi) - y))) / s2
        assert abs(got[f"grad_psi{i}"] - gr(x, *args)) <= TOL * scale
    assert abs(got["gradF_sigma"] - gsig(x, *args)) <= TOL * abs(gsig(x, *args))


@pytest.mark.parametrize("shape", [(243, 375), (240, 320)])
def test_setup_stage(sbd, O, cman, shape):
    """power iteration and observation synthesis with explicit randn, then with Philox (odd pixel count: the last
    element takes z0 of its pair)"""
    x = _crop(cman, shape)
    rng = np.random.default_rng(5)
    x0 = rng.standard_normal(shape)
    noise = rng.standard_normal(shape)
    cl = O.operators.closures(0, shape, 7, 0.0)
    eng = sbd.engine_for(shape, 7, 0, 0.0)
    val, iters = eng.max_eigenval((1.0, 1.0), 1e-4, 10000, x0=x0)
    want_val = O.metrics.max_eigenval(cl["A"], cl["AT"], (1.0, 1.0), shape, 1e-4, 10000, lambda s: x0)
    assert abs(val - want_val) <= 1e-11 * want_val and iters > 1
    # Philox start vector (stream 0xFFFF0001, step 0); at an odd pixel count the last element takes z0 of its pair
    val_p, _ = eng.max_eigenval((1.0, 1.0), 1e-4, 10000, seed=4)
    z0 = O.philox.randn_image(shape, 4, 0xFFFF0001, 0)
    want_p = O.metrics.max_eigenval(cl["A"], cl["AT"], (1.0, 1.0), shape, 1e-4, 10000, lambda s: z0)
    assert abs(val_p - want_p) <= 1e-11 * want_p
    y, sigma, nrm = eng.observe(x, PSI[0], 30, noise=noise)
    Ax = cl["A"](x, *PSI[0])
    want_sigma = np.linalg.norm(Ax - Ax.mean(), "fro") / np.sqrt(x.size * 10 ** 3.0)
    assert abs(sigma - want_sigma) <= 1e-12 * want_sigma
    assert rel(y, Ax + want_sigma * noise) < TOL
    # Philox: the noise of y is the oracle's counter-based stream (stream 0xFFFF0002, step 0)
    y2, sigma2, _ = eng.observe(x, PSI[0], 30, seed=9)
    z = O.philox.randn_image(shape, 9, 0xFFFF0002, 0)
    assert rel(y2, Ax + sigma2 * z) < TOL


def test_salsa_vs_oracle(sbd, O, cman):
    shape = (375, 375)              # odd side, square: the oracle's SALSA_v2 TV initialisation needs a square image
    x = _crop(cman, shape)
    cl = O.operators.closures(0, shape, 7, 0.0)
    rng = np.random.default_rng(3)
    y = cl["A"](x, *PSI[0]) + 2.0 * rng.standard_normal(shape)
    eng = sbd.engine_for(shape, 7, 0, 0.0)
    psi, tau, mu = PSI[0], 0.12, 0.003
    H = cl["H_FFT"](*psi)
    filt = 1.0 / (np.abs(H) ** 2 + mu)
    invLS = lambda z: np.real(O.operators._ifft2(filt * O.operators._fft2(z)))
    from oracle import salsa
    want = salsa.SALSA_v2(y, lambda z: cl["A"](z, *psi), tau, "MU", mu, "AT", lambda z: cl["AT"](z, *psi),
                            "StopCriterion", 1, "True_x", x, "ToleranceA", 1e-5, "MAXITERA", 12, "Phi", O.tv.TVnorm,
                            "TVINITIALIZATION", 1, "TViters", 10, "LS", invLS, "VERBOSE", 0)
    r = eng.salsa_tv(y, psi, tau, mu, maxiter=12, tolA=1e-5, tv_iters=10, x_true=x)
    assert rel(r["x"], want[0]) < 1e-9
    assert rel(r["objective"], np.ravel(want[3])[:r["n_outer"] + 1]) < 1e-10


# ---------------------------------------------------------------- SAPG
def _traj(got, want, names):
    for a_n, b_n in names:
        a, b = np.asarray(got[a_n]), np.asarray(want[b_n])
        assert a.shape == b.shape, (a_n, a.shape, b.shape)
        assert rel(a, b) < TRAJ_TOL, (a_n, rel(a, b))


def test_sapg_gaussian_240x320(sbd, O, cman):
    x = _crop(cman, (240, 320))
    tape = NoiseTape(21)
    y, op, c = O.operators.setup_demo(0, x, tape, samples=8, warmup=4, burnIn=5, fix_w1=0, fix_w2=0)
    tape.record = True
    th, w1, w2, s2, r = O.sapg.SAPG_algorithm_Guassian(y, op, c, tape)
    noise = np.stack(tape.tape)[:, None]
    _, _, _, _, g = sbd.SAPG_algorithm_Guassian(y, op, c, noise=noise)
    _traj(g, r, [(k, k) for k in ("thetas", "w1s", "w2s", "sigmas", "logPiTraceX", "gXTrace", "logPiTrace_WU", "err_psf")])
    assert rel(g["Xlast_sample"], r["Xlast_sample"]) < TRAJ_TOL


def test_sapg_moffat_243x375(sbd, O, boat):
    """odd rows: single-sweep prox (no fused or cooperative Chambolle kernel), odd pixel count"""
    x = _crop(boat, (243, 375))
    tape = NoiseTape(22)
    y, op = O.operators.setup_demo(1, x, tape, samples=6, warmup=3, burnIn=4)
    tape.record = True
    th, a, b, s2, r = O.sapg.SAPG_algorithm_moffat(y, op, tape)
    noise = np.stack(tape.tape)[:, None]
    _, _, _, _, g = sbd.SAPG_algorithm_moffat(y, op, noise=noise)
    _traj(g, r, [(k, k) for k in ("thetas", "alphas", "betas", "sigmas", "logPiTraceX", "gXTrace", "err_psf")])
    assert rel(g["Xlast_sample"], r["Xlast_sample"]) < TRAJ_TOL


def test_sapg_laplace_300x200(sbd, O, cman):
    x = _crop(cman, (300, 200))
    tape = NoiseTape(23)
    y, op = O.operators.setup_demo(2, x, tape, samples=8, warmup=4, burnIn=5)
    tape.record = True
    th, b, s2, r = O.sapg.SAPG_algorithm_laplace(y, op, tape)
    noise = np.stack(tape.tape)[:, None]
    _, _, _, g = sbd.SAPG_algorithm_laplace(y, op, noise=noise)
    _traj(g, r, [(k, k) for k in ("thetas", "bs", "sigmas", "logPiTraceX", "err_sample", "err_psf")])
    assert rel(g["X_sample"], r["X_sample"]) < TRAJ_TOL


def test_sapg_philox_two_chains_odd_pixels_and_post_mean(sbd, O, cman):
    """2 chains, Philox noise at an odd pixel count (the pairs of chain 1 straddle 16-byte boundaries)"""
    x = _crop(cman, (63, 75))
    tape = NoiseTape(24)
    y, op, c = O.operators.setup_demo(0, x, tape, samples=12, warmup=4, burnIn=8, fix_w1=0, fix_w2=0)
    nch, seed = 2, 31
    step = {}

    def randn_chain(ch, shape):
        s = step.get(ch, 0)
        step[ch] = s + 1
        return O.philox.randn_image(shape, seed, ch, s)

    want = O.sapg.sapg_multichain(0, y, op, c, randn_chain, nch)
    _, _, _, _, g = sbd.SAPG_algorithm_Guassian(y, op, c, n_chains=nch, seed=seed)
    assert rel(g["thetas"], want["thetas"]) < TRAJ_TOL
    assert rel(g["sigmas"], want["sigmas"]) < TRAJ_TOL
    for ch in range(nch):
        assert rel(g["Xlast_sample"][ch], want["X"][ch]) < TRAJ_TOL
    # posterior mean (one chain, noise tape) against the mean of the oracle's samples
    tape2 = NoiseTape(25)
    y, op, c = O.operators.setup_demo(0, x, tape2, samples=20, warmup=4, burnIn=8, fix_w1=0, fix_w2=0)
    tape2.record = True
    Xs = []
    op2 = dict(op)
    gradF = op["gradF"]

    def spy(X, *a):
        Xs.append(X.copy())
        return gradF(X, *a)

    op2["gradF"] = spy
    _, _, _, _, r = O.sapg.SAPG_algorithm_Guassian(y, op2, c, tape2)
    noise = np.stack(tape2.tape)[:, None]
    _, _, _, _, g = sbd.SAPG_algorithm_Guassian(y, op, c, noise=noise, post_mean=True)
    W, S, B = op["warmup"], op["samples"], op["burnIn"]
    main = Xs[(W - 1):] + [r["Xlast_sample"]]
    mmse = np.mean(np.stack(main[B:S]), axis=0)
    assert rel(g["posteriormean"], mmse) < TRAJ_TOL
    assert abs(O.metrics.PSNR(x, g["posteriormean"]) - O.metrics.PSNR(x, mmse)) < 0.01


# ---------------------------------------------------------------- sharding
SHARD_WORKER = textwrap.dedent("""
    import os, sys
    import numpy as np
    import torch, torch.distributed as dist
    sys.path.insert(0, sys.argv[1])
    import sbd_b200
    from sbd_b200 import host as H
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
    rows, cols, total = 480, 640, 4
    per = total // world
    x = np.load(sys.argv[2])
    eng = sbd_b200.Engine(rows, cols, 7, H.MOFFAT, 0.0, total, rank)
    Ax = eng.blur(x, (0.4, 3.5), H.OP_A)
    nrm = float(np.linalg.norm(Ax - Ax.mean()))
    sig = lambda b: nrm / np.sqrt(rows * cols * 10 ** (b / 10))
    y = Ax + sig(30) * np.random.default_rng(2).standard_normal((rows, cols))
    op = dict(samples=8, warmup=4, burnIn=5, psf_size=7, min_th=1e-3, max_th=1.0, th_init=0.01,
              alpha_init=1.0, beta_init=10.0, min_alpha=1e-2, max_alpha=1.0, min_beta=0.1, max_beta=10.0,
              alpha=0.4, beta=3.5, fix_alpha=0, fix_beta=0, fix_sigma=0, d_exp=0.8, d_scale=1.0,
              sigma=sig(30), sigma_init=(sig(18) ** 2 + sig(35) ** 2) / 2, sigma_min=sig(18) ** 2, sigma_max=sig(35) ** 2)
    Lf = min(0.993 ** 2 / op["sigma_min"], 0.993 ** 2 / op["sigma_max"])
    op["lambda"] = min(5 / Lf, 2.0); op["gamma"] = 0.98 / (Lf + 1 / op["lambda"])
    shard = sbd_b200.ChainShard(total, world, rank)
    shard.init_engine_comm(eng)
    prm = H.make_params(H.MOFFAT, op, None, n_chains=per, seed=7, chain_offset=shard.chain_offset, total_chains=total)
    out = eng.sapg(y, prm)
    keys = ("thetas", "sigmas", "psi0", "psi1", "logPiTraceX")
    mine = np.stack([out[k] for k in keys])
    sbd_b200._lib.lib.sbd_comm_destroy(eng._h)
    if rank == 0:
        ref = eng.sapg(y, H.make_params(H.MOFFAT, op, None, n_chains=total, seed=7, chain_offset=0, total_chains=total))
        print("bitwise:", np.array_equal(np.stack([ref[k] for k in keys]), mine))
    dist.barrier()
    dist.destroy_process_group()
    eng.close()
""")


def test_sharding_bit_identical(cman, tmp_path):
    """1 rank x 4 chains and 2 ranks x 2 chains at 480 x 640: bit-identical trajectories"""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    worker = tmp_path / "worker.py"
    worker.write_text(SHARD_WORKER)
    np.save(tmp_path / "x.npy", _crop(cman, (480, 640)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29611", str(worker), ROOT, str(tmp_path / "x.npy")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "bitwise: True" in r.stdout


# ---------------------------------------------------------------- Python and MATLAB surfaces
def test_run_demo_240x320(cman):
    from sbd_b200 import demo
    x = _crop(cman, (240, 320))
    res = demo.run_demo(0, x, samples=12, warmup=4, burnIn=8, map_estimate=True, use_graph=False, name="crop",
                        fix_w1=0, fix_w2=0)
    assert res["xMAP"].shape == x.shape and np.isfinite(res["mse"]) and res["salsa_outer"] >= 1
    assert np.all(np.isfinite(res["thetas"]))


def test_mex_gateway_non_pow2(O):
    sys.path.insert(0, os.path.join(ROOT, "tests", "mexrt"))
    import runtime as mex
    shape = (60, 45)
    x = np.random.default_rng(4).uniform(0, 255, shape)
    cl = O.operators.closures(0, shape, 7, 0.0)
    assert rel(mex.call_mex("blur", x, 0, 7, 0.0, [0.4, 0.3], 0)[0], cl["A"](x, 0.4, 0.3)) < TOL
    assert rel(mex.call_mex("blur", x, 0, 7, 0.0, [0.4, 0.3], 1)[0], cl["AT"](x, 0.4, 0.3)) < TOL
    want = O.psf.resize(O.psf.taps(0, 7, (0.4, 0.3), 0.0, 0), shape)
    assert rel(mex.call_mex("spectrum", [60, 45], 0, 7, 0.0, [0.4, 0.3], 0)[0], want) < TOL
