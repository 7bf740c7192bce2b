"""The fixed-geometry instance of the tensor-core K1 kernel (ber_tconv2.cuh: tconv2_geom; ber_host.cu: tconv2_fixed_geometry).

bench.py's headline shape (wtx, N = 256, 16 symbols, cp = 16, tail_tx = 8, L = 21, 16-QAM) runs "_hs", whose frame loop has
that geometry compiled in; every other shape of the fixed-shape class runs the class-only sibling "_hsc".  Both must count
exactly what the generic kernel counts: checked against the resolved twin (the generic kernel's code) on the same frames,
and against the debug-barrier build.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

import wofdm_b200 as W
from wofdm_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HS = "ber_f32t2_n256_t256_tiles9_b2_hs"


def headline(noise_norm=0, constellation=0, **kw):
    import bench
    c = dict(bench.CFG, noise_norm=noise_norm, constellation=constellation)
    s = W.params_from_name(c["system"], c["N"], c["cp"], c["tail_tx"], c["tail_rx"], bits=c["bits"], S=c["S"],
                           noise_norm=noise_norm, constellation=constellation, **kw)
    vt, vr = bench.windows_for(c, capi, s)
    return s, vt, vr


def test_headline_is_the_compiled_geometry():
    """ber_tconv2.cuh: TCV2_HS_WTX256 = {N, S, cp, cs, tail_tx, rm, shift, L, bits}"""
    import bench
    s, _, _ = headline()
    got = (s.N, s.S, s.cp, s.cs, s.tail_tx, s.tail_rx, s.rm, s.shift, bench.CFG["L"], s.bits)
    assert got == (256, 16, 16, 8, 8, 0, 16, 0, 21, 4)


# ---------------------------------------------------------------- GPU

@pytest.fixture(scope="module")
def handle():
    with W.Handle([0]) as h:
        yield h


def channels(C, L=21, seed=5):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((L, C)) + 1j * rng.standard_normal((L, C))) * np.exp(-np.arange(L) / 4.0)[:, None]


def kernel_of(handle, s, vt, vr, chans, snr):
    plan = handle.ber_plan(s, vt, vr, chans, snr)
    try:
        return plan.kernel
    finally:
        plan.close()


def same_counters_as_generic(handle, s, vt, vr, chans, snr, ens, seed, variant=0, shard=(0, 1)):
    got = handle.ber_run(s, vt, vr, chans, snr, ens, seed=seed, variant=variant, shard=shard)
    ref = handle.ber_run_resolved(s, [vt], [vr], chans, snr, ens, seed=seed, variant=variant, shard=shard,
                                  by_subcarrier=True, by_channel=True)
    assert np.array_equal(ref["sym_err"][0].sum(axis=(1, 2)), got["sym_err"]), (ref["sym_err"][0].sum(axis=(1, 2)), got["sym_err"])
    assert np.array_equal(ref["bit_err"][0].sum(axis=(1, 2)), got["bit_err"])
    assert got["sym_err"][0] > 0
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("noise_norm,constellation", [(0, 0), (1, 1), (0, 1), (1, 0)])
@pytest.mark.parametrize("seed,variant,shard", [(13, 2, (0, 1)), (7, 0, (1, 3))])
def test_headline_runs_the_geometry_instance_with_the_generic_counters(handle, noise_norm, constellation, seed, variant, shard):
    s, vt, vr = headline(noise_norm, constellation)
    chans = channels(5)
    snr = np.array([-5.0, 5.0, 15.0, 25.0])
    assert kernel_of(handle, s, vt, vr, chans, snr) == HS
    got = same_counters_as_generic(handle, s, vt, vr, chans, snr, 40, seed, variant, shard)
    assert np.all(np.diff(got["sym_err"]) <= 0)


@pytest.mark.gpu
def test_plain_rc_window_runs_the_geometry_instance(handle):
    s, _, vr = headline()
    vt = capi.rc_window_tx(s)
    chans = channels(4)
    snr = np.array([0.0, 10.0, 20.0])
    assert kernel_of(handle, s, vt, vr, chans, snr) == HS
    same_counters_as_generic(handle, s, vt, vr, chans, snr, 30, 21)


def class_shape(case):
    """shapes of the fixed-shape class one step off the compiled geometry"""
    L = 21
    if case == "cp32":
        s = W.params_from_name("wtx", 256, 32, 8, 0, bits=4, S=16)
    elif case == "s15":
        s = W.params_from_name("wtx", 256, 16, 8, 0, bits=4, S=15)
    elif case == "l20":
        s, L = W.params_from_name("wtx", 256, 16, 8, 0, bits=4, S=16), 20
    elif case in ("bits2", "bits6"):
        s = W.params_from_name("wtx", 256, 16, 8, 0, bits=int(case[-1]), S=16)
    else:
        raise ValueError(case)
    return s, capi.rc_window_tx(s), capi.rc_window_rx(s), L


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["cp32", "s15", "l20", "bits2", "bits6"])
@pytest.mark.parametrize("noise_norm,constellation", [(0, 0), (1, 1)])
def test_class_shapes_run_the_class_instance_with_the_generic_counters(handle, case, noise_norm, constellation):
    s, vt, vr, L = class_shape(case)
    s.noise_norm, s.constellation = noise_norm, constellation
    chans = channels(4, L=L)
    snr = np.array([0.0, 10.0, 20.0, 30.0])
    k = kernel_of(handle, s, vt, vr, chans, snr)
    assert k.startswith("ber_f32t2_n256_t256_tiles") and k.endswith("_b2_hsc"), k
    same_counters_as_generic(handle, s, vt, vr, chans, snr, 30, 17, variant=1)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["guard", "tx_window_not_flat", "rx_tails"])
def test_shapes_outside_the_class_run_neither(handle, case):
    chans = channels(3)
    snr = np.array([10.0, 30.0])
    if case == "guard":
        s, vt, vr = headline(guard=16)
    elif case == "tx_window_not_flat":
        s, vt, vr = headline()
        vt = vt.copy()
        vt[s.n_tx // 2] *= 0.99
    else:
        s = W.params_from_name("WOLA", 256, 16, 8, 10, bits=4, S=16)
        vt, vr = capi.rc_window_tx(s), capi.rc_window_rx(s)
    k = kernel_of(handle, s, vt, vr, chans, snr)
    assert k.startswith("ber_f32t2_n256_") and not k.endswith(("_hs", "_hsc")), k


CHILD = r"""
import sys, numpy as np
sys.path.insert(0, sys.argv[1])
import wofdm_b200 as W
from wofdm_b200 import capi
case = sys.argv[2]
if case == "headline":
    s = W.params_from_name("wtx", 256, 16, 8, 0, bits=4, S=16)
    L = 21
else:
    s = W.params_from_name("wtx", 256, 16, 8, 0, bits=4, S=15)
    L = 21
rng = np.random.default_rng(3)
chans = (rng.standard_normal((L, 4)) + 1j * rng.standard_normal((L, 4))) * np.exp(-np.arange(L) / 4.0)[:, None]
snr = np.array([0.0, 10.0, 20.0])
with W.Handle([0]) as h:
    vt, vr = capi.rc_window_tx(s), capi.rc_window_rx(s)
    p = h.ber_plan(s, vt, vr, chans, snr)
    print("KERNEL", p.kernel)
    p.close()
    r = h.ber_run(s, vt, vr, chans, snr, 40, seed=5, variant=3)
    print("COUNTERS", list(r["bit_err"]), list(r["sym_err"]))
"""


@pytest.mark.gpu
@pytest.mark.parametrize("case,kernel", [("headline", HS), ("s15", "ber_f32t2_n256_t256_tiles9_b2_hsc")])
def test_both_entries_against_debug_build(case, kernel):
    """libwofdm_dbg.so holds both entries with every relaxed synchronisation a full barrier: same counters"""
    dbg = os.path.join(ROOT, "w-ofdm-optimization_b200", "libwofdm_dbg.so")
    assert os.path.exists(dbg), "libwofdm_dbg.so is built by `make -C w-ofdm-optimization_b200/csrc` (__graft_entry__.build)"
    outs = []
    for lib in (None, dbg):
        env = dict(os.environ)
        env.pop("WOFDM_LIB", None)
        env.pop("WOFDM_VARIANT", None)
        if lib:
            env["WOFDM_LIB"] = lib
        r = subprocess.run([sys.executable, "-c", CHILD, ROOT, case], env=env, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
        assert f"KERNEL {kernel}\n" in r.stdout, r.stdout
        outs.append([l for l in r.stdout.splitlines() if l.startswith("COUNTERS")])
    assert outs[0] and outs[0] == outs[1], outs
