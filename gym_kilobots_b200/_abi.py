"""ctypes mirror of include/kb_b200.h (struct layouts, enums, function prototypes).

Shared by the product loader (`_native.py`, prefix ``kb_``, device pointers) and by the CPU
oracle wrapper used in tests (`oracle/kbo.py`, prefix ``kbo_``, host pointers).
"""
import ctypes as C

KB_MAX_POLY_VERTS = 8
KB_MAX_FIXTURES = 3
KB_MAX_LIGHTS = 4
KB_BODY_STATE_FLOATS = 12
KB_NUM_COUNTERS = 8

KB_SHAPE_CIRCLE, KB_SHAPE_POLYGON, KB_SHAPE_BOX = 0, 1, 2
KB_BODY_OBJECT = 0
KB_KILOBOT_PHOTOTAXIS = 1
KB_KILOBOT_SIMPLE_PHOTOTAXIS = 2
KB_KILOBOT_VELOCITY = 3
KB_KILOBOT_ACCELERATION = 4
KB_LIGHT_CIRCULAR, KB_LIGHT_MOMENTUM, KB_LIGHT_LINEAR = 1, 2, 3
KB_ACTION_NONE, KB_ACTION_LIGHT, KB_ACTION_KILOBOTS = 0, 1, 2

KB_STATUS_CONTACT_OVERFLOW = 1
KB_STATUS_NONFINITE = 2
KB_STATUS_SOLVER_OVERFLOW = 4

# task layer (extension beyond the reference, include/kb_b200.h "Task layer")
KB_TASK_CONST, KB_TASK_OBJECT_TO_TARGET, KB_TASK_SWARM_TO_TARGET = 0, 1, 2
KB_EPISODE_STATS = 6
KB_REDUCED_STATS = 8
REDUCED_STAT_NAMES = ("envs",) + ("return", "length", "position_error", "orientation_error", "success", "done_count") + ("envs_with_status",)
EPISODE_STAT_NAMES = ("return", "length", "position_error", "orientation_error", "success", "done_count")

COUNTER_NAMES = ("substeps", "contacts", "points", "levels", "pos_iters", "toi_events", "pair_tests", "islands")


class KbFixtureDef(C.Structure):
    _fields_ = [
        ("shape", C.c_int32),
        ("vertex_count", C.c_int32),
        ("radius", C.c_float),
        ("hx", C.c_float),
        ("hy", C.c_float),
        ("density", C.c_float),
        ("friction", C.c_float),
        ("restitution", C.c_float),
        ("vx", C.c_float * KB_MAX_POLY_VERTS),
        ("vy", C.c_float * KB_MAX_POLY_VERTS),
    ]


class KbBodyDef(C.Structure):
    _fields_ = [
        ("kind", C.c_int32),
        ("num_fixtures", C.c_int32),
        ("linear_damping", C.c_float),
        ("angular_damping", C.c_float),
        ("fixtures", KbFixtureDef * KB_MAX_FIXTURES),
    ]


class KbLightDef(C.Structure):
    _fields_ = [
        ("type", C.c_int32),
        ("relative_actions", C.c_int32),
        ("radius", C.c_double),
        ("bounds_lo", C.c_double * 2),
        ("bounds_hi", C.c_double * 2),
        ("action_lo", C.c_double * 2),
        ("action_hi", C.c_double * 2),
        ("max_velocity", C.c_double),
    ]


class KbSceneDesc(C.Structure):
    _fields_ = [
        ("num_bodies", C.c_int32),
        ("num_objects", C.c_int32),
        ("bodies", C.POINTER(KbBodyDef)),
        ("num_lights", C.c_int32),
        ("lights", C.POINTER(KbLightDef)),
        ("wall_x0", C.c_float),
        ("wall_y0", C.c_float),
        ("wall_x1", C.c_float),
        ("wall_y1", C.c_float),
        ("wall_edges", C.c_int32),
        ("wall_friction", C.c_float),
        ("steps_per_action", C.c_int32),
        ("velocity_iterations", C.c_int32),
        ("position_iterations", C.c_int32),
        ("dt", C.c_float),
        ("damping_mode", C.c_int32),
        ("enable_toi", C.c_int32),
        ("enable_sleep", C.c_int32),
        ("reward_const", C.c_float),
    ]


class KbDims(C.Structure):
    _fields_ = [
        ("num_envs", C.c_int32),
        ("num_bodies", C.c_int32),
        ("num_objects", C.c_int32),
        ("num_kilobots", C.c_int32),
        ("num_proxies", C.c_int32),
        ("max_contacts", C.c_int32),
        ("light_state_dim", C.c_int32),
        ("action_dim", C.c_int32),
        ("state_bytes_per_env", C.c_int32),
    ]


class KbTaskDef(C.Structure):
    _fields_ = [
        ("mode", C.c_int32),
        ("object", C.c_int32),
        ("max_episode_steps", C.c_int32),
        ("reserved", C.c_int32),
        ("w_position", C.c_double),
        ("w_orientation", C.c_double),
        ("step_penalty", C.c_double),
        ("success_bonus", C.c_double),
        ("position_tolerance", C.c_double),
        ("orientation_tolerance", C.c_double),
    ]


# per-kilobot local observations (include/kb_b200.h kb_local_observation)
KB_LOCAL_NEIGHBOURS, KB_LOCAL_OBJECTS, KB_LOCAL_LIGHT = 1, 2, 4


class KbLocalObsDef(C.Structure):
    _fields_ = [("radius", C.c_float), ("max_neighbours", C.c_int32), ("parts", C.c_int32), ("pad", C.c_int32)]


KB_SAMPLE_FIXED, KB_SAMPLE_RANDOM, KB_SAMPLE_AT_OBJECT = 0, 1, 2
KB_SAMPLE_MEAN_LIGHT, KB_SAMPLE_MEAN_RANDOM = 1, 2
KB_SAMPLE_MAX_OBJECTS = 16
KB_SAMPLE_MAX_CONFIGS = 16


class KbSampleObject(C.Structure):
    _fields_ = [("mode", C.c_int32), ("reserved", C.c_int32), ("pose", C.c_double * 3), ("extent", C.c_double)]


class KbSampleLight(C.Structure):
    _fields_ = [("mode", C.c_int32), ("reserved", C.c_int32), ("init", C.c_double * 2)]


class KbSampleSpec(C.Structure):
    _fields_ = [
        ("seed", C.c_uint64),
        ("env_id_base", C.c_int64),
        ("world_width", C.c_double),
        ("world_height", C.c_double),
        ("num_objects", C.c_int32),
        ("num_lights", C.c_int32),
        ("objects", C.POINTER(KbSampleObject)),
        ("lights", C.POINTER(KbSampleLight)),
        ("shuffle_lights", C.c_int32),
        ("kilobot_mean_mode", C.c_int32),
        ("perm_scene", C.POINTER(C.c_int32)),
        ("kilobot_mean", C.c_double * 2),
        ("kilobot_std", C.c_double),
    ]


# test-only geometry probe (include/kb_b200.h kb_probe_geometry)
KB_PROBE_SHAPE, KB_PROBE_COLLIDE, KB_PROBE_DISTANCE, KB_PROBE_TOI = 0, 1, 2, 3
KB_PROBE_OUT_WORDS = 40
KB_PROBE_FIXTURE, KB_PROBE_EDGE = 0, 1


class KbProbeShape(C.Structure):
    _fields_ = [("kind", C.c_int32), ("edge", C.c_int32), ("wall_edges", C.c_int32), ("wall_x0", C.c_float),
                ("wall_y0", C.c_float), ("wall_x1", C.c_float), ("wall_y1", C.c_float), ("fixture", KbFixtureDef)]


class KbProbeCase(C.Structure):
    _fields_ = [("a", C.c_int32), ("b", C.c_int32), ("fixed_rot_a", C.c_int32), ("fixed_rot_b", C.c_int32),
                ("xf_a", C.c_float * 4), ("xf_b", C.c_float * 4), ("sweep_a", C.c_float * 8), ("sweep_b", C.c_float * 8)]


# name -> (restype, argtypes); the exported symbol is prefix + name
_VP = C.c_void_p
PROTOTYPES = {
    "create": (C.c_int, [C.POINTER(KbSceneDesc), C.c_int32, _VP, C.c_int32, C.c_int32, C.c_int32, C.POINTER(_VP)]),
    "destroy": (C.c_int, [_VP]),
    "get_dims": (C.c_int, [_VP, C.POINTER(KbDims)]),
    "last_error": (C.c_char_p, []),
    "reset": (C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP]),
    "step": (C.c_int, [_VP, _VP, C.c_int32, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "step_host": (C.c_int, [_VP, _VP, C.c_int32, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "get_bodies": (C.c_int, [_VP, _VP]),
    "set_poses": (C.c_int, [_VP, _VP]),
    "set_poses_masked": (C.c_int, [_VP, _VP, _VP]),
    "get_status": (C.c_int, [_VP, _VP]),
    "set_env_scene": (C.c_int, [_VP, _VP]),
    "get_contacts": (C.c_int, [_VP, _VP, _VP]),
    "get_impulses": (C.c_int, [_VP, _VP]),
    "get_counters": (C.c_int, [_VP, _VP]),
    "get_proxies": (C.c_int, [_VP, _VP]),
    "get_controllers": (C.c_int, [_VP, _VP, _VP]),
    "get_mass_data": (C.c_int, [_VP, _VP]),
    "set_task": (C.c_int, [_VP, C.POINTER(KbTaskDef), _VP]),
    "get_episode_stats": (C.c_int, [_VP, _VP]),
    "bind_flat_observation": (C.c_int, [_VP, _VP]),
    "flat_observation_dim": (C.c_int, [_VP]),
    "render": (C.c_int, [_VP, _VP, C.c_int32, C.c_int32, C.c_int32, _VP, _VP]),
    "probe_geometry": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, _VP, C.c_int32, _VP, _VP]),
}
# exported by the product library only (the oracle has no state blob)
class KbLaunchConfig(C.Structure):
    _fields_ = [("lanes_per_env", C.c_int32), ("block_threads", C.c_int32), ("grid_blocks", C.c_int32),
                ("smem_bytes_per_block", C.c_int32), ("state_words_per_env", C.c_int32),
                ("smem_words_per_env", C.c_int32), ("specialised", C.c_int32), ("jit_ms", C.c_float),
                ("jit_reason", C.c_char * 256)]


PRODUCT_ONLY = {
    "get_body_counts": (C.c_int, [_VP, _VP, _VP]),
    "get_state": (C.c_int, [_VP, _VP]),
    "set_state": (C.c_int, [_VP, _VP]),
    "get_launch_config": (C.c_int, [_VP, C.POINTER(KbLaunchConfig)]),
    "jit_step_source": (C.c_int, [C.POINTER(KbSceneDesc), C.c_int32, C.c_int32, C.c_int32, C.c_char_p, C.c_int64,
                                  C.c_char_p, C.c_int64, C.POINTER(C.c_double)]),
    "get_host_layout": (C.c_int, [_VP, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "reduce_episode_stats": (C.c_int, [_VP, _VP, _VP]),
    "set_sampler": (C.c_int, [_VP, C.POINTER(KbSampleSpec)]),
    "set_sampler_mix": (C.c_int, [_VP, C.POINTER(KbSampleSpec), C.c_int32, _VP]),
    "current_scenes": (C.c_int, [_VP, _VP, _VP]),
    "reset_sampled": (C.c_int, [_VP, _VP, _VP]),
    "get_sampled": (C.c_int, [_VP, _VP, _VP, _VP, _VP]),
    "selftest_exact_math": (C.c_int, [C.c_int32, C.c_int32, C.POINTER(C.c_uint64)]),
    "local_observation_dim": (C.c_int, [_VP, C.POINTER(KbLocalObsDef)]),
    "local_observation": (C.c_int, [_VP, C.POINTER(KbLocalObsDef), _VP, _VP, _VP]),
}


def bind(lib, prefix, names=None):
    """Attach restype/argtypes to `lib` and return {name: function}."""
    out = {}
    table = dict(PROTOTYPES)
    if prefix == "kb_":
        table.update(PRODUCT_ONLY)
    for name, (res, args) in table.items():
        if names is not None and name not in names:
            continue
        fn = getattr(lib, prefix + name)
        fn.restype = res
        fn.argtypes = args
        out[name] = fn
    return out
