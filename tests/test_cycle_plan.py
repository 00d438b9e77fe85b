"""Host-side plan of a control cycle (`plan_cycle`, csrc/osc_launch.h), compiled for the host: which fused kernel (flag word) and
general path a cycle launches, and that every planned word is one of the declared instantiations.  The predicates the plan is
built from are tested in tests/test_launch_logic.py and tests/test_gain_selection.py.  No GPU needed: the functions only look at
the program struct."""
import ctypes as C
import itertools
import os
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
CUDA_INC = "/usr/local/cuda/include"

# flag word of the fused kernel (CV_* in osc_launch.h)
FULL, SPEC, GRAV, MOTION, PARK, PRG, F32 = (1 << k for k in range(7))
# GeneralPath
NONE, SINGULAR, BLEND, BLEND_SPLIT, GENERIC = range(5)
OSC_OK, OSC_ERR_UNSUPPORTED = 0, -2    # include/sai_b200_osc.h
MSG_F32_COVER = (b"FP32 mode covers a full six-dof MotionForceTask under pure motion control (alone or with a full JointTask) "
                 b"on an all-revolute-z chain only")
MSG_F32_GAINS = b"FP32 mode: the kernels have no single-precision form with per-robot gains (osc_set_gains)"

# program conditions of the probe's plan() (enum Cond in tests/cpp/cycle_plan_probe.cpp)
C_FULL, C_OFF_AXIS, C_TWO_CLAMPED, C_FORCE, C_CLOSED_LOOP, C_VEL_SAT = 1, 2, 4, 8, 16, 32
C_MFT_GAINS, C_JT_GAINS, C_GRAVITY, C_SPLIT_HINT, C_SCRATCH, C_FP32 = 64, 128, 256, 512, 1024, 2048


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    if not os.path.exists(os.path.join(CUDA_INC, "cuda_runtime.h")):
        pytest.skip("CUDA headers not installed")
    out = tmp_path_factory.mktemp("plan") / "libcycle_plan_probe.so"
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-fPIC", "-shared", "-I", CUDA_INC, "-o", str(out), os.path.join(HERE, "cpp", "cycle_plan_probe.cpp")])
    lib = C.CDLL(str(out))
    lib.plan.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_uint), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_char_p)]
    return lib


def run_plan(probe, n, R, has_jt, cond):
    word, general, launches, msg = C.c_uint(), C.c_int(), C.c_int(), C.c_char_p()
    err = probe.plan(n, R, int(has_jt), cond, C.byref(word), C.byref(general), C.byref(launches), C.byref(msg))
    if err != OSC_OK:
        return err, msg.value
    return err, word.value, general.value, launches.value


def declared(probe, R, f32=False):
    out = (C.c_uint * 16)()
    count = probe.cycle_words(R, int(f32), out)
    assert 0 < count <= 16
    return list(out[:count])


def test_flag_bits(probe):
    out = (C.c_uint * 7)()
    probe.cycle_bits(out)
    assert list(out) == [FULL, SPEC, GRAV, MOTION, PARK, PRG, F32]


# ---- equivalence with the parent commit's launch decision --------------------------------------------------------------
# What commit 1c4c694 launched, restated independently of osc_launch.h: the FP32 gate of run_cycle (osc_capi.cu:1539-1547), the
# kernel ladder of launch_one (osc_cycle_kernels.cu:95-150, template defaults of launch_variant at :42), its general-path choice
# (osc_cycle_kernels.cu:152-211, the general hierarchy at :240) and the launch count of run_cycle (osc_capi.cu:1610).

def variant(full, spec=False, grav=False, motion=None, park=False, prg=False):
    """the word of launch_variant<N, R, JT, FULL, SPEC, GRAV, MOTION = SPEC, PARK, PRG>"""
    motion = spec if motion is None else motion
    return (FULL if full else 0) | (SPEC if spec else 0) | (GRAV if grav else 0) | (MOTION if motion else 0) | (PARK if park else 0) | (PRG if prg else 0)


def prg_specialised(R, spec, motion):
    """cycle_prg_specialised, osc_launch.h:103"""
    return spec and ((R == 6 and motion) or R == 3)


def parent_plan(n, R, has_jt, cond):
    full = R != 0 and (6 if R < 0 else R) == 6 and bool(cond & C_FULL)    # the probe's program: P.mft[0].full
    mft_leads = R != 0
    # cycle_spec_eligible (osc_launch.h:65-94) on the probe's programs: an all-revolute-z chain with light links and a full
    # joint task without velocity saturation, unless a condition breaks it
    spec = not (cond & (C_OFF_AXIS | C_TWO_CLAMPED))
    motion = full and not (cond & (C_FORCE | C_CLOSED_LOOP | C_VEL_SAT))            # mft_pure_motion (osc_launch.h:55-61)
    grav = bool(cond & C_GRAVITY)
    fp32 = bool(cond & C_FP32)
    # cycle_per_robot_gains (osc_launch.h:97-99)
    prg = (mft_leads and bool(cond & C_MFT_GAINS)) or (has_jt and bool(cond & C_JT_GAINS))
    # blend_split_selected (osc_launch.h:31-34): pipelined handle, grid hint not "small", rank = 6 (R < 0: the probe's six-dof task)
    split = bool(cond & C_SPLIT_HINT) and not fp32 and bool(cond & C_SCRATCH) and mft_leads and full

    # run_cycle, osc_capi.cu:1539-1547
    if fp32:
        if not (R == 6 and full and spec and motion and n == 7):    # fused_f32_available: n == 7
            return OSC_ERR_UNSUPPORTED, MSG_F32_COVER
        if cond & (C_MFT_GAINS | C_JT_GAINS):
            return OSC_ERR_UNSUPPORTED, MSG_F32_GAINS
    if R < 0:    # osc_cycle_kernels.cu:240, osc_capi.cu:1610
        return OSC_OK, 0, GENERIC, 1

    # launch_one, osc_cycle_kernels.cu:98-150
    if R == 6:
        park = full and split
        if fp32:
            w = F32 | variant(True, True, grav, True)      # launch_f32<N, JT, GRAV>, osc_cycle_f32.cu:14-40
        elif not full:
            w = variant(False)
        elif prg and prg_specialised(R, spec, motion):
            w = variant(True, True, grav, True, park, True)
        elif prg and not park:
            w = variant(True)
        elif prg:
            w = variant(True, False, False, False, True)
        elif spec and motion and not park:
            w = variant(True, True, grav)
        elif spec and motion:
            w = variant(True, True, grav, True, True)
        elif spec and not park:
            w = variant(True, True, grav, False)
        elif spec:
            w = variant(True, True, grav, False, True)
        elif not park:
            w = variant(True)
        else:
            w = variant(True, False, False, False, True)
    elif R == 3:
        if spec and prg and prg_specialised(R, spec, motion):
            w = variant(False, True, grav, False, False, True)
        elif spec:
            w = variant(False, True, grav, False)
        else:
            w = variant(False)
    elif R == 0:
        w = variant(False, prg=True) if prg else variant(False)
    else:
        w = variant(False)

    # osc_cycle_kernels.cu:152-211
    if R == 0:
        general = NONE
    elif R == 6 and full and split:
        general = BLEND_SPLIT
    elif R == 6 and full:
        general = BLEND
    else:
        general = SINGULAR
    launches = (4 if split else 2) if R > 0 else 1    # osc_capi.cu:1610
    return OSC_OK, w, general, launches


LAWS = [0, C_FORCE, C_CLOSED_LOOP, C_VEL_SAT]
BREAKERS = [0, C_OFF_AXIS, C_TWO_CLAMPED]
GAINS = [0, C_MFT_GAINS, C_JT_GAINS, C_MFT_GAINS | C_JT_GAINS]
HINTS = [0, C_SPLIT_HINT, C_SCRATCH, C_SPLIT_HINT | C_SCRATCH]


def test_plan_matches_parent_ladder_and_declared_lists(probe):
    lists = {R: set(declared(probe, R)) for R in range(-1, 7)}
    f32_list = set(declared(probe, 6, True))
    planned = {R: set() for R in range(-1, 7)}
    planned_f32 = set()
    count = 0
    for n, R, has_jt, full, breaker, law, gains, grav, hint, fp32 in itertools.product(
            [4, 6, 7, 8], range(-1, 7), [False, True], [0, C_FULL], BREAKERS, LAWS, GAINS, [0, C_GRAVITY], HINTS, [0, C_FP32]):
        cond = full | breaker | law | gains | grav | hint | fp32
        got = run_plan(probe, n, R, has_jt, cond)
        want = parent_plan(n, R, has_jt, cond)
        assert got == want, (n, R, has_jt, cond)
        count += 1
        if got[0] != OSC_OK or R < 0:
            continue
        if got[1] & F32:
            assert R == 6 and got[1] & ~F32 in f32_list, (n, R, has_jt, cond, got)
            planned_f32.add(got[1] & ~F32)
        else:
            assert got[1] in lists[R], (n, R, has_jt, cond, got)
            planned[R].add(got[1])
    assert count == 4 * 8 * 2 * 2 * 3 * 4 * 4 * 2 * 4 * 2
    # the lists hold no instantiation the planner never asks for
    assert planned_f32 == f32_list
    for R in range(0, 7):
        assert planned[R] == lists[R], R
    assert len(lists[6]) == 15 and len(lists[3]) == 5 and len(lists[0]) == 2 and lists[1] == {0} and len(f32_list) == 2
