"""ctypes binding of include/dqn_zoo_b200.h (the C ABI).  No compute happens in Python.

The CUDA library is mandatory: importing this module raises if it is missing, and every
entry point raises on a non-zero status.  There is no CPU fallback anywhere in the package.
"""

import ctypes as C
import os

from dqn_zoo_b200 import _build

i32, i64, f32, f64, u64 = C.c_int32, C.c_int64, C.c_float, C.c_double, C.c_uint64
vp = C.c_void_p

DZ_FLAG_BAD_VALUE, DZ_FLAG_BAD_INDEX, DZ_FLAG_BAD_TARGET, DZ_FLAG_ROOT_ZERO, DZ_FLAG_NONFINITE_WEIGHT = 1, 2, 4, 8, 16
DZ_FLAG_FRAME_POOL_FULL = 32
DZ_FRAME_WINDOW, DZ_FRAME_MAX_STACK, DZ_FRAME_MAX_STAGE_BYTES = 16, 8, 200 * 1024
AGENT_KINDS = {'dqn': 0, 'double_q': 1, 'prioritized': 2, 'c51': 3, 'qrdqn': 4, 'rainbow': 5, 'iqn': 6}
OPTIMIZERS = {'adam': 0, 'rmsprop': 1}


class FrameStore(C.Structure):
  _fields_ = [('d_frames', vp), ('d_row_frames', vp), ('d_frame_hash', vp), ('d_frame_born', vp),
              ('d_frame_last_ref', vp), ('d_state', vp), ('d_add_stage', vp), ('d_batch_stage', vp), ('num_frames', i64),
              ('frame_bytes', i64), ('frame_stride', i64), ('stack', i32), ('batch_capacity', i32)]


class ReplayView(C.Structure):
  _fields_ = [('d_obs', vp), ('d_action', vp), ('d_reward', vp), ('d_discount', vp), ('capacity', i64),
              ('obs_bytes', i64), ('obs_stride', i64), ('d_tree', vp), ('first_leaf', i64), ('d_live', vp),
              ('d_id_at', vp), ('d_ids', vp), ('d_flags', vp), ('frames', FrameStore)]


class AddRecord(C.Structure):
  _fields_ = [('slot', i64), ('action', i32), ('reward', f64), ('discount', f64), ('n_patches', i32),
              ('patch_pos', i64 * 4), ('patch_val', i64 * 4), ('patch_target', i32 * 4), ('tree_index', i64),
              ('leaf_value', f64), ('evict_index', i64), ('size_after', i64), ('d_priority', vp), ('alpha', f64),
              ('item_id', i64), ('oldest_live', i64)]


class SampleInputs(C.Structure):
  _fields_ = [('d_rand_pos', vp), ('d_u_tree', vp), ('d_u_mix', vp), ('d_scalars', vp)]


class SampleOutputs(C.Structure):
  _fields_ = [('d_ids', vp), ('d_indices', vp), ('d_slots', vp), ('d_probs', vp), ('d_weights', vp)]


class LearnerConfig(C.Structure):
  _fields_ = [('kind', i32), ('num_actions', i32), ('num_atoms', i32), ('num_quantiles', i32), ('latent_dim', i32),
              ('tau_samples_s_tm1', i32), ('tau_samples_policy', i32), ('tau_samples_s_t', i32), ('batch', i32),
              ('obs_h', i32), ('obs_w', i32), ('obs_c', i32), ('vmax', f32), ('grad_error_bound', f32),
              ('huber_param', f32), ('optimizer', i32), ('learning_rate', f32), ('opt_eps', f32), ('rms_decay', f32),
              ('adam_b1', f32), ('adam_b2', f32), ('max_global_grad_norm', f32)]


class LearnerPlan(C.Structure):
  _fields_ = [('param_count', i64), ('num_tensors', i32), ('opt_state_floats', i64), ('workspace_bytes', i64),
              ('noise_floats', i64), ('tau_floats', i64)]


class LearnerBuffers(C.Structure):
  _fields_ = [('d_online', vp), ('d_target', vp), ('d_grads', vp), ('d_opt_state', vp), ('d_workspace', vp),
              ('d_counters', vp)]


class Batch(C.Structure):
  _fields_ = [('d_s_tm1_rows', vp), ('d_s_t_rows', vp), ('d_a_tm1', vp), ('d_r_t', vp), ('d_discount_t', vp),
              ('d_weights', vp), ('d_taus', vp), ('d_noise', vp)]


class UpdateOutputs(C.Structure):
  _fields_ = [('d_loss', vp), ('d_per_example', vp), ('d_priorities', vp), ('d_grad_norm', vp)]


class ResampleAxis(C.Structure):   # struct dz_resample_axis
  _fields_ = [('d_bounds', C.c_void_p), ('d_kk', C.c_void_p), ('ksize', C.c_int32), ('in_size', C.c_int32),
              ('out_size', C.c_int32)]


class LearnIO(C.Structure):
  _fields_ = [('sample_in', SampleInputs), ('sample_out', SampleOutputs), ('d_taus', vp), ('d_noise', vp),
              ('update_out', UpdateOutputs), ('d_max_seen_priority', vp), ('priority_exponent', f64)]


class DzError(RuntimeError):
  pass


_ERRORS = {-1: ValueError, -2: DzError, -3: IndexError, -4: DzError}

_SIGNATURES = {
    'dz_last_error': (C.c_char_p, []),
    'dz_build_info': (C.c_char_p, []),
    'dz_launch_count': (i64, []),
    'dz_profile_begin': (i32, []),
    'dz_profile_end': (i32, [C.c_char_p, i64]),
    'dz_sumtree_rebuild': (i32, [vp, i64, i64, vp]),
    'dz_sumtree_set': (i32, [vp, i64, i64, vp, vp, i64, vp, vp]),
    'dz_sumtree_query': (i32, [vp, i64, vp, i64, vp, vp, vp]),
    'dz_sumtree_get': (i32, [vp, i64, i64, vp, i64, vp, vp, vp]),
    'dz_replay_add': (i32, [C.POINTER(ReplayView), C.POINTER(AddRecord), vp, vp, vp]),
    'dz_replay_fill_synthetic': (i32, [C.POINTER(ReplayView), i64, i64, u64, i32, f64, vp]),
    'dz_replay_fill_synthetic_frames': (i32, [C.POINTER(ReplayView), i64, i64, u64, i32, f64, vp]),
    'dz_test_frame_hash': (i32, [vp, i64, vp]),
    'dz_replay_sample': (i32, [C.POINTER(ReplayView), i32, C.POINTER(SampleInputs), C.POINTER(SampleOutputs), i32, vp]),
    'dz_replay_gather': (i32, [C.POINTER(ReplayView), vp, i32, vp, vp, vp, vp, vp, vp]),
    'dz_replay_update_priorities': (i32, [C.POINTER(ReplayView), vp, vp, i32, f64, i64, vp]),
    'dz_learner_plan_query': (i32, [C.POINTER(LearnerConfig), C.POINTER(LearnerPlan)]),
    'dz_learner_tensor_info': (i32, [C.POINTER(LearnerConfig), i32, C.c_char_p, C.POINTER(i64), C.POINTER(i32),
                                     C.POINTER(i64)]),
    'dz_learner_create': (i32, [C.POINTER(LearnerConfig), C.POINTER(LearnerBuffers), C.POINTER(vp)]),
    'dz_learner_destroy': (None, [vp]),
    'dz_learner_update': (i32, [vp, C.POINTER(Batch), C.POINTER(UpdateOutputs), i32, vp]),
    'dz_learner_learn': (i32, [vp, C.POINTER(ReplayView), i32, C.POINTER(LearnIO), vp]),
    'dz_learner_generate_randomness': (i32, [vp, u64, vp, vp, vp]),
    'dz_learner_generate_randomness_async': (i32, [vp, u64, vp, vp, vp]),
    'dz_learner_q_values': (i32, [vp, vp, vp, vp, vp, vp]),
    'dz_learner_act_batch': (i32, [vp, vp, i32, vp, vp, vp, f32, vp, vp, vp]),
    'dz_learner_sync_target': (i32, [vp, vp]),
    'dz_test_u8_to_unit': (i32, [vp, vp]),
    'dz_atari_preprocess': (i32, [vp, vp, i32, vp, vp, vp, vp, i32, vp, i32, vp]),
    'dz_atari_preprocess_band_rows': (i32, []),
    'dz_jax_uniform': (i32, [vp, vp, i32, vp, vp]),
    'dz_test_threefry2x32': (i32, [C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, vp]),
    'dz_test_learner_buffer': (i32, [vp, C.c_char_p, vp, vp]),
    'dz_test_copy': (i32, [vp, vp, i64, vp]),
    'dz_test_learner_trace': (i32, [vp, C.c_char_p, vp]),
    'dz_debug_timeline': (i32, [vp]),
    'dz_test_tc_pgemm_work': (i64, [i32, i32, i32]),
    'dz_test_tc_pgemm': (i32, [vp, i32, i32, i32, vp, i32, i32, i32, i32, i32, vp, vp, i64, i64, i32, i64, vp, i32, vp]),
    'dz_test_umma_gemm': (i32, [vp, i32, vp, i32, i32, i32, i32, i32, vp, i32, i32, vp, i32, vp, vp, vp, vp]),
}

EXPORTS = tuple(_SIGNATURES)


def library_path():
  return _build.LIB_PATH


def _load():
  path = library_path()
  if not os.path.exists(path):
    raise ImportError('dqn_zoo_b200: %s is missing — run `python -c "import __graft_entry__ as g; g.build()"` '
                      '(there is no CPU fallback)' % path)
  lib = C.CDLL(path)
  for name, (res, args) in _SIGNATURES.items():
    fn = getattr(lib, name)
    fn.restype, fn.argtypes = res, args
  return lib


lib = _load()


def check(status):
  if status != 0:
    raise _ERRORS.get(status, DzError)(lib.dz_last_error().decode())


def call(name, *args):
  check(getattr(lib, name)(*args))
