"""numpy mirrors of the POD structs in include/ismpc_b200.h (layout checked by tests/test_abi.py).

Host-side plumbing only: these dtypes describe the byte layout of the batch arrays that cross the
C ABI.  Field names follow the reference (AMR_code_DART/types.hpp:7-81, parameters.cpp:9-45,
trotting/quad_as_bip_bang.m:25-58).
"""
import numpy as np

MAX_FSTEPS = 8

STATE = np.dtype([("com_pos", "f8", 3), ("com_vel", "f8", 3), ("zmp_pos", "f8", 3)], align=True)
WALK = np.dtype([("sim_time", "f8"), ("mpc_iter", "i4"), ("control_iter", "i4"),
                 ("footstep_counter", "i4"), ("support_foot", "i4")], align=True)
FORMC_MODEL = np.dtype([("dt", "f8"), ("dtc", "f8"), ("mass", "f8"), ("g", "f8"),
                        ("q_p", "f8"), ("q_v", "f8"), ("q_u", "f8"), ("fz_max", "f8"),
                        ("N", "i4"), ("reserved", "i4")], align=True)
FORMC_INST = np.dtype([("com_height", "f8"), ("box_w", "f8"), ("box_w_init", "f8"),
                       ("S", "i4"), ("F_ds", "i4"), ("plan_first_row", "i4"), ("n_steps", "i4")], align=True)
FORMC_OUT = np.dtype([("next", STATE), ("zmp_in", "f8", 2), ("fz0", "f8"), ("lambda0", "f8"),
                      ("kkt_res", "f8"), ("status", "i4"), ("iters", "i4", 3)], align=True)
FORMC_TICK = np.dtype([("state", STATE), ("walk", WALK), ("reserved", "f8", 4)], align=True)      # ismpc_formc_tick_t, 128 bytes
FORMA_MODEL = np.dtype([("dt", "f8"), ("g_eta", "f8"), ("q_zdot", "f8"), ("q_foot", "f8"),
                        ("disp_forw", "f8"), ("disp_forw_dummy", "f8"), ("disp_L", "f8"),
                        ("C", "i4"), ("P", "i4"), ("F", "i4"), ("reserved", "i4")], align=True)
FORMA_INST = np.dtype([("st", "f8", 6), ("cur_fs", "f8", 2), ("fs_store", "f8", 2), ("height", "f8"),
                       ("wx", "f8"), ("wy", "f8"), ("j", "i4"), ("fs_counter", "i4"), ("ds", "i4"),
                       ("cl_first_ramp", "i4"), ("timing_first", "i4"), ("n_timing", "i4"),
                       ("plan_first_row", "i4"), ("n_fs", "i4")], align=True)
FORMA_OUT = np.dtype([("st", "f8", 6), ("pred_fs", "f8", 2 * MAX_FSTEPS), ("kkt_res", "f8"),
                      ("status", "i4"), ("iters", "i4")], align=True)
FORMA_GRAD = np.dtype([("st", "f8", 6), ("cur_fs", "f8", 2), ("fs_store", "f8", 2), ("height", "f8"), ("wx", "f8"),
                       ("wy", "f8"), ("status", "i4"), ("reserved", "i4")], align=True)      # ismpc_forma_grad_t
PUSH = np.dtype([("fs", "i4"), ("ct0", "i4"), ("ct1", "i4"), ("reserved", "i4"),
                 ("ax", "f8"), ("ay", "f8")], align=True)

FEET_MODEL = np.dtype([("disp_forw", "f8"), ("disp_i", "f8"), ("disp_o", "f8"), ("disp_forw_dummy", "f8"),
                       ("disp_i_dummy", "f8"), ("disp_o_dummy", "f8"), ("gait", "i4"), ("wrap_counter", "i4")], align=True)
FEET_INST = np.dtype([("phi", "f8"), ("j", "i4"), ("fs_counter", "i4"), ("timing_first", "i4"), ("n_timing", "i4"),
                      ("plan_first_row", "i4"), ("plan_rows", "i4")], align=True)
GAIT_TROT, GAIT_WALK = 0, 1
PLAN_MODEL = np.dtype([("disp_B", "f8"), ("disp_C", "f8"), ("disp_forw", "f8"), ("disp_i", "f8"), ("disp_o", "f8"),
                       ("gait", "i4"), ("N_gait", "i4")], align=True)
PLAN_REQ = np.dtype([("disp_A", "f8"), ("phi", "f8")], align=True)
KF_MODEL = np.dtype([("h_com", "f4"), ("mass", "f4"), ("sampling_time", "f4"), ("g", "f4"),
                     ("q_process", "f4", (3, 4)), ("q_measurement", "f4", (3, 9))], align=True)
KF_STATE = np.dtype([("state", "f4", (3, 5)), ("sigma", "f4", (3, 25))], align=True)
KF_SAMPLE = np.dtype([("meas", "f4", (3, 3)), ("input", "f4", 3)], align=True)
KF_STATE64 = np.dtype([("state", "f8", (3, 5)), ("sigma", "f8", (3, 25))], align=True)

SIZES = {"ismpc_state_t": 72, "ismpc_walk_t": 24, "ismpc_formc_model_t": 72, "ismpc_formc_inst_t": 40,
         "ismpc_formc_out_t": 128, "ismpc_formc_tick_t": 128, "ismpc_forma_model_t": 72, "ismpc_forma_inst_t": 136,
         "ismpc_forma_out_t": 192, "ismpc_forma_grad_t": 112, "ismpc_push_t": 32, "ismpc_feet_model_t": 56, "ismpc_feet_inst_t": 32, "ismpc_plan_model_t": 48, "ismpc_plan_req_t": 16, "ismpc_kf_model_t": 172, "ismpc_kf_state_t": 360,
         "ismpc_kf_sample_t": 48, "ismpc_kf_state64_t": 720}
DTYPES = {"ismpc_state_t": STATE, "ismpc_walk_t": WALK, "ismpc_formc_model_t": FORMC_MODEL,
          "ismpc_formc_inst_t": FORMC_INST, "ismpc_formc_out_t": FORMC_OUT, "ismpc_formc_tick_t": FORMC_TICK,
          "ismpc_forma_model_t": FORMA_MODEL, "ismpc_forma_inst_t": FORMA_INST,
          "ismpc_forma_out_t": FORMA_OUT, "ismpc_forma_grad_t": FORMA_GRAD, "ismpc_push_t": PUSH, "ismpc_feet_model_t": FEET_MODEL,
          "ismpc_feet_inst_t": FEET_INST, "ismpc_plan_model_t": PLAN_MODEL, "ismpc_plan_req_t": PLAN_REQ,
          "ismpc_kf_model_t": KF_MODEL, "ismpc_kf_state_t": KF_STATE, "ismpc_kf_sample_t": KF_SAMPLE, "ismpc_kf_state64_t": KF_STATE64}

# status bits
ST_OK, ST_Z_FAIL, ST_X_FAIL, ST_Y_FAIL, ST_WINDOW, ST_XY_SKIPPED, ST_NAN_GUARD, ST_QP_FAIL = 0, 1, 2, 4, 8, 16, 32, 64
ST_GI_FALLBACK = 128    # informational: form-A result came from the dual active-set fallback
ST_FAIL_MASK = ST_Z_FAIL | ST_X_FAIL | ST_Y_FAIL | ST_WINDOW | ST_QP_FAIL
MEM_HOST, MEM_DEVICE, MEM_HOST_ASYNC = 0, 1, 2


def formc_model(dt=0.01, dtc=0.01, mass=50.0, g=9.81, q_p=1005000.0, q_v=100.0, q_u=0.01,
                fz_max=10000.0, N=100):
    """Reference constants: AMR_code_DART/parameters.cpp:9-45, MPCSolver.cpp:159,253-255."""
    m = np.zeros(1, dtype=FORMC_MODEL)
    m["dt"], m["dtc"], m["mass"], m["g"] = dt, dtc, mass, g
    m["q_p"], m["q_v"], m["q_u"], m["fz_max"], m["N"] = q_p, q_v, q_u, fz_max, N
    return m


def forma_model(dt=0.01, g_eta=9.8, q_zdot=1.0, q_foot=1e7, disp_forw=0.5, disp_forw_dummy=0.25,
                disp_L=0.4, C=100, P=200, F=3):
    """Reference constants: trotting/quad_as_bip_bang.m:11,25-31,239-240; init_quadruped.m:31-36."""
    m = np.zeros(1, dtype=FORMA_MODEL)
    m["dt"], m["g_eta"], m["q_zdot"], m["q_foot"] = dt, g_eta, q_zdot, q_foot
    m["disp_forw"], m["disp_forw_dummy"], m["disp_L"] = disp_forw, disp_forw_dummy, disp_L
    m["C"], m["P"], m["F"] = C, P, F
    return m


def feet_model(gait, disp_forw=0.5, disp_i=0.4, disp_o=0.4, wrap_counter=0):
    """Reference constants: trotting/init_quadruped.m:31-36 == walking/init_quadruped2.m:31-36."""
    m = np.zeros(1, dtype=FEET_MODEL)
    m["disp_forw"], m["disp_i"], m["disp_o"] = disp_forw, disp_i, disp_o
    m["disp_forw_dummy"], m["disp_i_dummy"], m["disp_o_dummy"] = disp_forw / 2, disp_i / 2, disp_o / 2
    m["gait"] = GAIT_TROT if gait in ("trot", GAIT_TROT) else GAIT_WALK
    m["wrap_counter"] = wrap_counter
    return m


def plan_model(gait, N_gait=100, disp_B=0.259394, disp_C=0.88, disp_forw=0.5, disp_i=0.4, disp_o=0.4):
    """Reference constants: trotting/init_quadruped.m:4-36 == walking/init_quadruped2.m:4-36."""
    m = np.zeros(1, dtype=PLAN_MODEL)
    m["disp_B"], m["disp_C"], m["disp_forw"], m["disp_i"], m["disp_o"] = disp_B, disp_C, disp_forw, disp_i, disp_o
    m["gait"] = GAIT_TROT if gait in ("trot", GAIT_TROT) else GAIT_WALK
    m["N_gait"] = N_gait
    return m


def kf_model(h_com=0.69, mass=50.0, sampling_time=0.01, g=9.81, q_process=1e-2, q_measurement=1e-4):
    """StateFiltering's constructor arguments (AMR_code_DART/StateFiltering.hpp:19-22); the reference never
    instantiates the class, so the noise covariances have no reference values: diagonal defaults."""
    m = np.zeros(1, dtype=KF_MODEL)
    m["h_com"], m["mass"], m["sampling_time"], m["g"] = h_com, mass, sampling_time, g
    m["q_process"][0] = np.tile((np.eye(2) * q_process).reshape(-1), (3, 1))
    m["q_measurement"][0] = np.tile((np.eye(3) * q_measurement).reshape(-1), (3, 1))
    return m


def pack_ticks(state, walk):
    """ismpc_formc_tick_t records from the state / walk arrays of a batch."""
    t = np.zeros(len(state), dtype=FORMC_TICK)
    t["state"] = state; t["walk"] = walk
    return t
