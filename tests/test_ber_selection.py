"""Which K1 kernel each BER entry point prepares, pinned as a table (ber_host.cu: choose_variant, choose_resolved).

Every row is an entry point and a shape; the expected value is the WOFDM_DEBUG residency report of prepare_kernel for the
one kernel the call prepares: "<name>: smem <bytes> B, <n> CTAs/SM".  So a row fixes the kernel, its shared-memory layout and its
residency on a B200.  Plans prepare their kernel without running it; the other calls run one or two tiny frames.
"""
import re

import numpy as np
import pytest

import wofdm_b200 as W
from oracle import wofdm_oracle as O

pytestmark = pytest.mark.gpu

ENV = ("WOFDM_DEBUG", "WOFDM_NO_TCONV", "WOFDM_NO_CIRC", "WOFDM_VARIANT", "WOFDM_RESOLVED_STAGED", "WOFDM_MASK_FFT",
       "WOFDM_MASK_DUMP", "WOFDM_MAX_CTAS_PER_SM")

# (system, N, cp, tail_tx, tail_rx, S, L, precision, guard, window pairs, flat Tx window, environment)
SHAPES = {
    # the fixed-shape class (ber_tconv2.cuh: HS) and one shape just outside each of its conditions
    "hs": ("wtx", 256, 16, 8, 0, 16, 21, 0, 0, 1, True, {}),
    "hs_2pairs": ("wtx", 256, 16, 8, 0, 16, 21, 0, 0, 2, True, {}),
    "hs_tail_rx": ("WOLA", 256, 16, 8, 10, 16, 21, 0, 0, 1, True, {}),
    "hs_guard": ("wtx", 256, 16, 8, 0, 16, 21, 0, 64, 1, True, {}),
    "hs_not_flat": ("wtx", 256, 16, 8, 0, 16, 21, 0, 0, 1, False, {}),
    "hs_cs_short": ("CPwtx", 256, 16, 8, 0, 16, 21, 0, 0, 1, True, {}),
    # tensor-core kernels: N = 256 / 512 / 1024, L = 21 / 84, several pairs in one launch
    "tconv_n256_3pairs": ("WOLA", 256, 16, 8, 10, 16, 21, 0, 0, 3, True, {}),
    "tconv_n256_l84": ("WOLA", 256, 16, 8, 10, 16, 84, 0, 0, 2, True, {}),
    "tconv_n512": ("CPW", 512, 32, 16, 20, 16, 21, 0, 0, 2, True, {}),
    "tconv_n512_l84": ("CPW", 512, 32, 16, 20, 16, 84, 0, 0, 1, True, {}),
    "tconv_n1024": ("WOLA", 1024, 64, 32, 40, 16, 21, 0, 0, 1, True, {}),
    "tconv_n1024_l84": ("CPW", 1024, 64, 32, 40, 16, 84, 0, 0, 2, True, {}),
    # several pairs at a shape without a tensor-core kernel: one launch per pair
    "pairs_s7": ("WOLA", 256, 30, 8, 10, 7, 21, 0, 0, 2, True, {}),
    # register kernels
    "regs_exact_fit": ("WOLA", 256, 16, 8, 10, 16, 21, 0, 0, 1, True, {"WOFDM_NO_TCONV": "1"}),
    "regs_circ": ("wrx", 256, 16, 0, 10, 16, 21, 0, 0, 1, True, {"WOFDM_NO_TCONV": "1"}),
    "regs_c19_circ": ("wtx", 256, 32, 8, 0, 16, 21, 0, 0, 1, True, {"WOFDM_NO_TCONV": "1"}),
    "regs_c19": ("wtx", 256, 32, 8, 0, 16, 21, 0, 0, 1, False, {"WOFDM_NO_TCONV": "1"}),
    "regs_c19_no_circ": ("wtx", 256, 32, 8, 0, 16, 21, 0, 0, 1, True, {"WOFDM_NO_TCONV": "1", "WOFDM_NO_CIRC": "1"}),
    "regs_n512": ("WOLA", 512, 32, 16, 20, 16, 21, 0, 0, 2, True, {"WOFDM_NO_TCONV": "1"}),
    "regs_n1024_cluster": ("CPW", 1024, 64, 32, 40, 16, 21, 0, 0, 2, True, {"WOFDM_NO_TCONV": "1"}),
    # staged kernels; frames that do not fit shared memory keep their buffers in global memory
    "staged_n64": ("WOLA", 64, 8, 4, 4, 16, 5, 0, 0, 2, True, {}),
    "staged_n1024_s48": ("WOLA", 1024, 64, 32, 40, 48, 21, 0, 0, 1, True, {}),
    "fp64_n256": ("WOLA", 256, 16, 8, 10, 16, 21, 1, 0, 2, True, {}),
    "fp64_n1024": ("WOLA", 1024, 64, 32, 40, 16, 21, 1, 0, 1, True, {}),
    # the staged twin with production's noise numbering
    "resolved_staged": ("WOLA", 256, 16, 8, 10, 16, 21, 0, 0, 1, True, {"WOFDM_RESOLVED_STAGED": "1"}),
    "resolved_staged_regs": ("WOLA", 256, 16, 8, 10, 16, 21, 0, 0, 1, True, {"WOFDM_RESOLVED_STAGED": "1", "WOFDM_NO_TCONV": "1"}),
}
PLAN_CALLS = ("plan", "resolved", "segments")

# (system, N, cp, tail_tx, tail_rx, S, L, guard, environment) of the channel-mask chain
MASKED = {
    "gather_n256": ("wtx", 256, 16, 8, 0, 16, 21, 64, {}),
    "gather_n512": ("CPW", 512, 32, 16, 20, 16, 21, 128, {}),
    "mask_fft_n256": ("wtx", 256, 16, 8, 0, 16, 21, 64, {"WOFDM_MASK_FFT": "1"}),
    "l84_n256": ("wtx", 256, 16, 8, 0, 16, 30, 64, {}),
    "regs_txs_s7": ("WOLA", 256, 30, 8, 10, 7, 21, 64, {}),
    "staged_s48": ("wtx", 256, 16, 8, 0, 48, 21, 0, {}),
    "resolved_staged": ("wtx", 256, 16, 8, 0, 16, 21, 64, {"WOFDM_RESOLVED_STAGED": "1"}),
}
MASKED_CALLS = ("masked", "masked_resolved")

# wofdm_ber_verify: its four kernel kinds
VERIFY = {
    "n256_wrx": ("wrx", 256, 16, 0, 10, 16, 21, 0),
    "n1024": ("WOLA", 1024, 64, 32, 40, 16, 21, 0),
}
VERIFY_CALLS = ("verify", "verify_staged", "verify_direct", "verify_no_tconv")

ROWS = ([f"{k}/{c}" for k in SHAPES for c in PLAN_CALLS] + [f"masked_{k}/{c}" for k in MASKED for c in MASKED_CALLS] +
        [f"verify_{k}/{c}" for k in VERIFY for c in VERIFY_CALLS])

# recorded on a B200 (148 SMs, 227 KB of shared memory per block)
EXPECTED = {
    "hs/plan": "ber_f32t2_n256_t256_tiles9_b2_hs: smem 92528 B, 2 CTAs/SM",
    "hs/resolved": "ber_f32t2_n256_t256_tiles9_b2_cl1_lTCV_LB_res: smem 94576 B, 2 CTAs/SM",
    "hs/segments": "ber_f32t2_n256_t256_tiles9_b2_cl1_lTCV_LB_res: smem 94576 B, 2 CTAs/SM",
    "hs_2pairs/plan": "ber_f32t2_n256_t256_tiles9_b2: smem 94672 B, 2 CTAs/SM",
    "hs_2pairs/resolved": "ber_f32t2_n256_t256_tiles9_b2_cl1_lTCV_LB_res: smem 98768 B, 2 CTAs/SM",
    "hs_2pairs/segments": "ber_f32t2_n256_t256_tiles9_b2_cl1_lTCV_LB_res: smem 98768 B, 2 CTAs/SM",
    "hs_tail_rx/plan": "ber_f32t2_n256_t256_tiles9_b2: smem 92576 B, 2 CTAs/SM",
    "hs_tail_rx/resolved": "ber_f32t2_n256_t256_tiles9_b2_cl1_lTCV_LB_res: smem 94624 B, 2 CTAs/SM",
    "hs_tail_rx/segments": "ber_f32t2_n256_t256_tiles9_b2_cl1_lTCV_LB_res: smem 94624 B, 2 CTAs/SM",
    "hs_guard/plan": "ber_f32t2_n256_t256_tiles9_b2: smem 92528 B, 2 CTAs/SM",
    "hs_guard/resolved": "ber_f32t2_n256_t256_tiles9_b2_cl1_lTCV_LB_res: smem 94576 B, 2 CTAs/SM",
    "hs_guard/segments": "ber_f32t2_n256_t256_tiles9_b2_cl1_lTCV_LB_res: smem 94576 B, 2 CTAs/SM",
    "hs_not_flat/plan": "ber_f32t2_n256_t256_tiles9_b2: smem 92528 B, 2 CTAs/SM",
    "hs_not_flat/resolved": "ber_f32t2_n256_t256_tiles9_b2_cl1_lTCV_LB_res: smem 94576 B, 2 CTAs/SM",
    "hs_not_flat/segments": "ber_f32t2_n256_t256_tiles9_b2_cl1_lTCV_LB_res: smem 94576 B, 2 CTAs/SM",
    "hs_cs_short/plan": "ber_f32t2_n256_t256_tiles9_b2: smem 92496 B, 2 CTAs/SM",
    "hs_cs_short/resolved": "ber_f32t2_n256_t256_tiles9_b2_cl1_lTCV_LB_res: smem 94544 B, 2 CTAs/SM",
    "hs_cs_short/segments": "ber_f32t2_n256_t256_tiles9_b2_cl1_lTCV_LB_res: smem 94544 B, 2 CTAs/SM",
    "tconv_n256_3pairs/plan": "ber_f32t2_n256_t256_tiles9_b2: smem 96960 B, 2 CTAs/SM",
    "tconv_n256_3pairs/resolved": "ber_f32t2_n256_t256_tiles9_b2_cl1_lTCV_LB_res: smem 103104 B, 2 CTAs/SM",
    "tconv_n256_3pairs/segments": "ber_f32t2_n256_t256_tiles9_b2_cl1_lTCV_LB_res: smem 103104 B, 2 CTAs/SM",
    "tconv_n256_l84/plan": "ber_f32t2_n256_t256_tiles9_b2_cl1_l84: smem 103472 B, 2 CTAs/SM",
    "tconv_n256_l84/resolved": "ber_f32t2_n256_t256_tiles9_b2_cl1_l84_res: smem 107568 B, 2 CTAs/SM",
    "tconv_n256_l84/segments": "ber_f32t2_n256_t256_tiles9_b2_cl1_l84_res: smem 107568 B, 2 CTAs/SM",
    "tconv_n512/plan": "ber_f32t2_n512_t512_tiles18_b1: smem 183696 B, 1 CTAs/SM",
    "tconv_n512/resolved": "ber_f32t2_n512_t512_tiles18_b1_cl1_lTCV_LB_res: smem 191888 B, 1 CTAs/SM",
    "tconv_n512/segments": "ber_f32t2_n512_t512_tiles18_b1_cl1_lTCV_LB_res: smem 191888 B, 1 CTAs/SM",
    "tconv_n512_l84/plan": "ber_f32_n512_t256_c0_l0_b1_ffalse: smem 170000 B, 1 CTAs/SM",
    "tconv_n512_l84/resolved": "ber_f32_n512_t256_c0_l0_b1_f0_res: smem 174096 B, 1 CTAs/SM",
    "tconv_n512_l84/segments": "ber_f32_n512_t256_c0_l0_b1_f0_res: smem 174096 B, 1 CTAs/SM",
    "tconv_n1024/plan": "ber_f32t2_n1024_t512_tiles18_b1_cl2: smem 192816 B, 1 CTAs/SM",
    "tconv_n1024/resolved": "ber_f32t2_n1024_t512_tiles18_b1_cl2_lTCV_LB_res: smem 201008 B, 1 CTAs/SM",
    "tconv_n1024/segments": "ber_f32t2_n1024_t512_tiles18_b1_cl2_lTCV_LB_res: smem 201008 B, 1 CTAs/SM",
    "tconv_n1024_l84/plan": "ber_f32t2_n1024_t512_tiles18_b1_cl2_l84: smem 210416 B, 1 CTAs/SM",
    "tconv_n1024_l84/resolved": "ber_f32t2_n1024_t512_tiles18_b1_cl2_l84_res: smem 226800 B, 1 CTAs/SM",
    "tconv_n1024_l84/segments": "ber_f32t2_n1024_t512_tiles18_b1_cl2_l84_res: smem 226800 B, 1 CTAs/SM",
    "pairs_s7/plan": "ber_f32r_n256_t256_c17_l21_b2_ffalse: smem 69328 B, 2 CTAs/SM",
    "pairs_s7/resolved": "ber_f32r_n256_t256_c17_l21_b2_ffalse_cl1_res: smem 71376 B, 2 CTAs/SM",
    "pairs_s7/segments": "ber_f32r_n256_t256_c17_l21_b2_ffalse_cl1_res: smem 71376 B, 2 CTAs/SM",
    "regs_exact_fit/plan": "ber_f32r_n256_t256_c17_l21_b2_ftrue: smem 88016 B, 2 CTAs/SM",
    "regs_exact_fit/resolved": "ber_f32r_n256_t256_c17_l21_b2_ftrue_cl1_res: smem 90064 B, 2 CTAs/SM",
    "regs_exact_fit/segments": "ber_f32r_n256_t256_c17_l21_b2_ftrue_cl1_res: smem 90064 B, 2 CTAs/SM",
    "regs_circ/plan": "ber_f32r_n256_t256_c19_l21_b2_ffalse_circ: smem 94128 B, 2 CTAs/SM",
    "regs_circ/resolved": "ber_f32r_n256_t256_c19_l21_b2_ffalse_cl1_circ_res: smem 96176 B, 2 CTAs/SM",
    "regs_circ/segments": "ber_f32r_n256_t256_c19_l21_b2_ffalse_cl1_circ_res: smem 96176 B, 2 CTAs/SM",
    "regs_c19_circ/plan": "ber_f32r_n256_t256_c19_l21_b2_ffalse_circ: smem 94144 B, 2 CTAs/SM",
    "regs_c19_circ/resolved": "ber_f32r_n256_t256_c19_l21_b2_ffalse_cl1_circ_res: smem 96192 B, 2 CTAs/SM",
    "regs_c19_circ/segments": "ber_f32r_n256_t256_c19_l21_b2_ffalse_cl1_circ_res: smem 96192 B, 2 CTAs/SM",
    "regs_c19/plan": "ber_f32r_n256_t256_c19_l21_b2_ffalse: smem 94144 B, 2 CTAs/SM",
    "regs_c19/resolved": "ber_f32r_n256_t256_c19_l21_b2_ffalse_cl1_res: smem 96192 B, 2 CTAs/SM",
    "regs_c19/segments": "ber_f32r_n256_t256_c19_l21_b2_ffalse_cl1_res: smem 96192 B, 2 CTAs/SM",
    "regs_c19_no_circ/plan": "ber_f32r_n256_t256_c19_l21_b2_ffalse: smem 94144 B, 2 CTAs/SM",
    "regs_c19_no_circ/resolved": "ber_f32r_n256_t256_c19_l21_b2_ffalse_cl1_res: smem 96192 B, 2 CTAs/SM",
    "regs_c19_no_circ/segments": "ber_f32r_n256_t256_c19_l21_b2_ffalse_cl1_res: smem 96192 B, 2 CTAs/SM",
    "regs_n512/plan": "ber_f32r_n512_t512_c17_l21_b1_ftrue: smem 174736 B, 1 CTAs/SM",
    "regs_n512/resolved": "ber_f32r_n512_t512_c17_l21_b1_ftrue_cl1_res: smem 178832 B, 1 CTAs/SM",
    "regs_n512/segments": "ber_f32r_n512_t512_c17_l21_b1_ftrue_cl1_res: smem 178832 B, 1 CTAs/SM",
    "regs_n1024_cluster/plan": "ber_f32r_n1024_t512_c19_l21_b1_ffalse_cl2: smem 204688 B, 1 CTAs/SM",
    "regs_n1024_cluster/resolved": "ber_f32r_n1024_t512_c19_l21_b1_ffalse_cl2_res: smem 212880 B, 1 CTAs/SM",
    "regs_n1024_cluster/segments": "ber_f32r_n1024_t512_c19_l21_b1_ffalse_cl2_res: smem 212880 B, 1 CTAs/SM",
    "staged_n64/plan": "ber_f32_n64_t64_c0_l0_b1_ffalse: smem 23888 B, 4 CTAs/SM",
    "staged_n64/resolved": "ber_f32_n64_t64_c0_l0_b1_f0_res: smem 24400 B, 4 CTAs/SM",
    "staged_n64/segments": "ber_f32_n64_t64_c0_l0_b1_f0_res: smem 24400 B, 4 CTAs/SM",
    "staged_n1024_s48/plan": "ber_f32_n1024_t512_c0_l0_b1_ffalse: smem 155088 B, 1 CTAs/SM",
    "staged_n1024_s48/resolved": "ber_f32_n1024_t512_c0_l0_b1_f0_res: smem 163280 B, 1 CTAs/SM",
    "staged_n1024_s48/segments": "ber_f32_n1024_t512_c0_l0_b1_f0_res: smem 163280 B, 1 CTAs/SM",
    "fp64_n256/plan": "ber_f64_n256_t256_c0_l0_b1_ffalse: smem 166784 B, 1 CTAs/SM",
    "fp64_n256/resolved": "ber_f64_n256_t256_c0_l0_b1_f0_res: smem 168832 B, 1 CTAs/SM",
    "fp64_n256/segments": "ber_f64_n256_t256_c0_l0_b1_f0_res: smem 168832 B, 1 CTAs/SM",
    "fp64_n1024/plan": "ber_f64_n1024_t256_c0_l0_b1_ffalse: smem 152224 B, 1 CTAs/SM",
    "fp64_n1024/resolved": "ber_f64_n1024_t256_c0_l0_b1_f0_res: smem 160416 B, 1 CTAs/SM",
    "fp64_n1024/segments": "ber_f64_n1024_t256_c0_l0_b1_f0_res: smem 160416 B, 1 CTAs/SM",
    "resolved_staged/plan": "ber_f32t2_n256_t256_tiles9_b2: smem 92576 B, 2 CTAs/SM",
    "resolved_staged/resolved": "ber_f32_n256_t256_c0_l0_b1_f0_res: smem 87872 B, 1 CTAs/SM",
    "resolved_staged/segments": "ber_f32_n256_t256_c0_l0_b1_f0_res: smem 87872 B, 1 CTAs/SM",
    "resolved_staged_regs/plan": "ber_f32r_n256_t256_c17_l21_b2_ftrue: smem 88016 B, 2 CTAs/SM",
    "resolved_staged_regs/resolved": "ber_f32_n256_t256_c0_l0_b1_f0_res: smem 87872 B, 1 CTAs/SM",
    "resolved_staged_regs/segments": "ber_f32_n256_t256_c0_l0_b1_f0_res: smem 87872 B, 1 CTAs/SM",
    "masked_gather_n256/masked": "ber_f32t2_n256_t256_tiles9_b2_txy: smem 92528 B, 2 CTAs/SM",
    "masked_gather_n256/masked_resolved": "ber_f32t2_n256_t256_tiles9_b2_txy_res: smem 94576 B, 2 CTAs/SM",
    "masked_gather_n512/masked": "ber_f32t2_n512_t512_tiles18_b1_txy: smem 179280 B, 1 CTAs/SM",
    "masked_gather_n512/masked_resolved": "ber_f32t2_n512_t512_tiles18_b1_txy_res: smem 183376 B, 1 CTAs/SM",
    "masked_mask_fft_n256/masked": "ber_f32t2_n256_t256_tiles9_b2: smem 92528 B, 2 CTAs/SM",
    "masked_mask_fft_n256/masked_resolved": "ber_f32t2_n256_t256_tiles9_b2_cl1_lTCV_LB_res: smem 94576 B, 2 CTAs/SM",
    "masked_l84_n256/masked": "ber_f32t2_n256_t256_tiles9_b2_cl1_l84: smem 101232 B, 2 CTAs/SM",
    "masked_l84_n256/masked_resolved": "ber_f32t2_n256_t256_tiles9_b2_cl1_l84_res: smem 103280 B, 2 CTAs/SM",
    "masked_regs_txs_s7/masked": "ber_f32r_n256_t256_c17_l21_b2_ffalse_txs: smem 69328 B, 2 CTAs/SM",
    "masked_regs_txs_s7/masked_resolved": "ber_f32r_n256_t256_c17_l21_b2_ffalse_txs_res: smem 71376 B, 2 CTAs/SM",
    "masked_staged_s48/masked": "ber_f32_n256_t256_c0_l0_b1_ffalse: smem 231184 B, 1 CTAs/SM",
    "masked_staged_s48/masked_resolved": "ber_f32_n256_t256_c0_l0_b1_f0_res: smem 60944 B, 1 CTAs/SM",
    "masked_resolved_staged/masked": "ber_f32t2_n256_t256_tiles9_b2_txy: smem 92528 B, 2 CTAs/SM",
    "masked_resolved_staged/masked_resolved": "ber_f32_n256_t256_c0_l0_b1_f0_res: smem 87824 B, 1 CTAs/SM",
    "verify_n256_wrx/verify": "ber_f32t2_n256_t256_tiles9_b2_verify: smem 92576 B, 2 CTAs/SM",
    "verify_n256_wrx/verify_staged": "ber_f32_n256_t256_c0_l0_b1_ffalse_verify: smem 86400 B, 1 CTAs/SM",
    "verify_n256_wrx/verify_direct": "ber_f32r_n256_t256_c19_l21_b2_ffalse_verify: smem 94128 B, 2 CTAs/SM",
    "verify_n256_wrx/verify_no_tconv": "ber_f32r_n256_t256_c19_l21_b2_ffalse_circ_verify: smem 94128 B, 2 CTAs/SM",
    "verify_n1024/verify": "ber_f32t2_n1024_t512_tiles18_b1_cl2_verify: smem 192816 B, 1 CTAs/SM",
    "verify_n1024/verify_staged": "ber_f32_n1024_t512_c0_l0_b1_ffalse_verify: smem 122320 B, 1 CTAs/SM",
    "verify_n1024/verify_direct": "ber_f32r_n1024_t512_c17_l21_b1_ftrue_cl2_verify: smem 192544 B, 1 CTAs/SM",
    "verify_n1024/verify_no_tconv": "ber_f32r_n1024_t512_c17_l21_b1_ftrue_cl2_verify: smem 192544 B, 1 CTAs/SM",
}


@pytest.fixture(scope="module")
def handle():
    with W.Handle([0]) as h:
        yield h


def system(name, N, cp, ttx, trx, S, precision=0, guard=0):
    p = O.system_params(name, N, cp, ttx, trx, S=S, bits=4, guard=guard)
    s = W.SysT(N=p.N, cp=p.cp, cs=p.cs, tail_tx=p.tail_tx, tail_rx=p.tail_rx, rm=p.rm, shift=p.shift, bits=p.bits, S=p.S,
               noise_norm=0, constellation=0, precision=precision, guard=p.guard)
    return p, s


def windows(p, pairs, flat=True):
    wins = [O.perturbed_windows(p, seed=p.N + k)[:2] for k in range(pairs - 1)] + [(O.rc_window_tx(p), O.rc_window_rx(p))]
    wt, wr = [w[0].copy() for w in wins], [w[1] for w in wins]
    if not flat:
        for w in wt:
            w[p.n_tx // 2] *= 0.99
    return wt, wr


def env_of(row):
    shape, call = row.split("/")
    if call in PLAN_CALLS:
        return SHAPES[shape][-1]
    return MASKED[shape[len("masked_"):]][-1] if call in MASKED_CALLS else {}


def run(handle, row):
    shape, call = row.split("/")
    snr = np.array([10.0])
    if call in PLAN_CALLS:
        name, N, cp, ttx, trx, S, L, prec, guard, pairs, flat, _ = SHAPES[shape]
        p, s = system(name, N, cp, ttx, trx, S, prec, guard)
        wt, wr = windows(p, pairs, flat)
        chans = O.synth_channels(1, L, seed=1)
        if call == "plan":
            plan = handle.ber_plan_multi(s, wt, wr, chans, snr) if pairs > 1 else handle.ber_plan(s, wt[0], wr[0], chans, snr)
            plan.close()
        elif call == "resolved":
            handle.ber_run_resolved(s, wt, wr, chans, snr, 1, by_subcarrier=True, by_channel=False)
        else:
            handle.ber_run_segments(s, wt, wr, chans, snr, 2, [(0, 1, 1)])
    elif call in MASKED_CALLS:
        name, N, cp, ttx, trx, S, L, guard, _ = MASKED[shape[len("masked_"):]]
        p, s = system(name, N, cp, ttx, trx, S, 0, guard)
        vt, vr, _, _ = O.perturbed_windows(p, seed=N + cp)
        chans = O.synth_channels(1, L, seed=1)
        if call == "masked":
            handle.ber_run_masked(s, vt, vr, chans, snr, 1)
        else:
            handle.ber_run_masked_resolved(s, vt, vr, chans, snr, 1, by_subcarrier=True, by_channel=False)
    else:
        name, N, cp, ttx, trx, S, L, prec = VERIFY[shape[len("verify_"):]]
        p, s = system(name, N, cp, ttx, trx, S, prec)
        chans = O.synth_channels(1, L, seed=1)
        sym, nz = handle.ber_draws(s, L, 3, 0, [0])
        handle.ber_verify(s, O.rc_window_tx(p), O.rc_window_rx(p), chans, snr, sym, nz, force_staged=call == "verify_staged",
                          direct=call == "verify_direct", no_tconv=call == "verify_no_tconv")


def prepared(handle, row, monkeypatch, capfd):
    """the residency reports of the kernels the call of `row` prepared"""
    for k in ENV:
        monkeypatch.delenv(k, raising=False)
    for k, v in env_of(row).items():
        monkeypatch.setenv(k, v)
    monkeypatch.setenv("WOFDM_DEBUG", "1")
    capfd.readouterr()
    run(handle, row)
    return re.findall(r"\[wofdm\] (\S+: smem \d+ B, \d+ CTAs/SM)", capfd.readouterr().err)


@pytest.mark.parametrize("row", ROWS)
def test_selection(handle, row, monkeypatch, capfd):
    assert prepared(handle, row, monkeypatch, capfd) == [EXPECTED[row]], row
