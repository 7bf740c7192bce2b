"""The fixed-shape instance of the tensor-core K1 kernel (ber_tconv2.cuh: HS; ber_host.cu: tconv2_fixed_shape).

Jobs with a flat Tx window (cp, cs >= tail_tx), no Rx window tails, one window pair, no guard band and the symbols drawn in
the kernel run an instance whose frame loop has those switches as constants.  It must count exactly what the generic
kernel counts: checked against the resolved twin, which stays generic, on the same frames, and against the debug-barrier
build.  Every other shape keeps the generic kernel.

CPU: bench.py's headline windows are in the class.  GPU: selection, counters, debug build.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

import wofdm_b200 as W
from wofdm_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def headline(noise_norm=0, constellation=0, **kw):
    """bench.py's configs[1] system and its windows (RC tails perturbed by a seeded +-10 %)."""
    import bench
    c = dict(bench.CFG, noise_norm=noise_norm, constellation=constellation)
    s = W.params_from_name(c["system"], c["N"], c["cp"], c["tail_tx"], c["tail_rx"], bits=c["bits"], S=c["S"],
                           noise_norm=noise_norm, constellation=constellation, **kw)
    vt, vr = bench.windows_for(c, capi, s)
    return s, vt, vr


def flat_tx(s, vt):
    """ber_host.cu: flat_tx_window."""
    body = vt[s.tail_tx:s.n_tx - s.tail_tx]
    return s.cp >= s.tail_tx and s.cs >= s.tail_tx and body[0] != 0 and bool(np.all(body == body[0]))


def test_headline_windows_are_in_the_class():
    s, vt, vr = headline()
    assert flat_tx(s, vt) and s.tail_rx == 0 and s.guard == 0
    assert not np.all(vt[:s.tail_tx] == vt[s.tail_tx])          # (the tails themselves are windowed)


# ---------------------------------------------------------------- GPU

@pytest.fixture(scope="module")
def handle():
    with W.Handle([0]) as h:
        yield h


def channels(C, L=21, seed=5):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((L, C)) + 1j * rng.standard_normal((L, C))) * np.exp(-np.arange(L) / 4.0)[:, None]


def kernel_of(handle, s, vt, vr, chans, snr, multi=False):
    plan = handle.ber_plan_multi(s, vt, vr, chans, snr) if multi else handle.ber_plan(s, vt, vr, chans, snr)
    try:
        return plan.kernel
    finally:
        plan.close()


@pytest.mark.gpu
@pytest.mark.parametrize("noise_norm,constellation", [(0, 0), (1, 1)])
def test_headline_job_runs_the_fixed_instance_with_the_generic_counters(handle, noise_norm, constellation):
    """configs[1]-shaped jobs, python and MATLAB conventions: the plan runs the fixed-shape instance, and its counters equal,
    bit for bit, the sums of the resolved twin (the generic kernel's code with per-cell counters) on the same frames."""
    s, vt, vr = headline(noise_norm, constellation)
    chans = channels(6)
    snr = np.array([-5.0, 5.0, 15.0, 25.0])
    ens = 50                                                  # 1200 frames, 4.6e6 decisions
    assert kernel_of(handle, s, vt, vr, chans, snr) == "ber_f32t2_n256_t256_tiles9_b2_hs"
    got = handle.ber_run(s, vt, vr, chans, snr, ens, seed=13, variant=2)
    ref = handle.ber_run_resolved(s, [vt], [vr], chans, snr, ens, seed=13, variant=2, by_subcarrier=True, by_channel=True)
    assert np.array_equal(ref["sym_err"][0].sum(axis=(1, 2)), got["sym_err"]), (ref["sym_err"][0].sum(axis=(1, 2)), got["sym_err"])
    assert np.array_equal(ref["bit_err"][0].sum(axis=(1, 2)), got["bit_err"])
    assert got["sym_err"][0] > 0 and np.all(np.diff(got["sym_err"]) <= 0)
    # the plain RC window is in the class too
    assert kernel_of(handle, s, capi.rc_window_tx(s), vr, chans, snr).endswith("_hs")


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["guard", "two_pairs", "tx_window_not_flat", "rx_tails", "short_prefix"])
def test_shapes_outside_the_class_run_the_generic_kernel(handle, case):
    chans = channels(3)
    snr = np.array([10.0, 30.0])
    multi = False
    if case == "guard":
        s, vt, vr = headline(guard=16)
    elif case == "two_pairs":
        s, vt, vr = headline()
        vt, vr, multi = [vt, vt * 0.9], [vr, vr], True
    elif case == "tx_window_not_flat":
        s, vt, vr = headline()
        vt = vt.copy()
        vt[s.n_tx // 2] *= 0.99
    elif case == "rx_tails":
        s = W.params_from_name("WOLA", 256, 16, 8, 10, bits=4, S=16)
        vt, vr = capi.rc_window_tx(s), capi.rc_window_rx(s)
    else:                                                      # cp < tail_tx: the window's head is not inside the prefix
        s = W.params_from_name("wtx", 256, 4, 8, 0, bits=4, S=16)
        vt, vr = capi.rc_window_tx(s), capi.rc_window_rx(s)
    k = kernel_of(handle, s, vt, vr, chans, snr, multi)
    assert k.startswith("ber_f32t2_n256_") and not k.endswith("_hs"), k


@pytest.mark.gpu
def test_fixed_instance_against_debug_build():
    """As test_ber_gpu.py::test_relaxed_barriers_against_debug_build, on a job the fixed-shape instance runs: libwofdm_dbg.so
    holds that instance with every relaxed synchronisation a full barrier, and the counters must be identical."""
    dbg = os.path.join(ROOT, "w-ofdm-optimization_b200", "libwofdm_dbg.so")
    assert os.path.exists(dbg), "libwofdm_dbg.so is built by `make -C w-ofdm-optimization_b200/csrc` (__graft_entry__.build)"
    outs = []
    for lib in (None, dbg, None):
        env = dict(os.environ)
        env.pop("WOFDM_LIB", None)
        if lib:
            env["WOFDM_LIB"] = lib
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "sanitize_k1.py"), "wtx"], env=env, capture_output=True,
                           text=True, timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
        assert "KERNEL ber_f32t2_n256_t256_tiles9_b2_hs" in r.stdout, r.stdout
        outs.append([l for l in r.stdout.splitlines() if l.startswith("COUNTERS")])
    assert outs[0] and outs[0] == outs[1] == outs[2], outs
