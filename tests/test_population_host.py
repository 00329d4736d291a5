"""Population training without a GPU: the config rules of a population and the argument checks of the grouped ops
(brl_ppo_grad_grouped, brl_mlp_adam_step_grouped), which run before any CUDA work."""
import ctypes

import pytest


def _config(**kw):
    c = dict(num_envs=64, num_steps=4, minibatch_size=64, update_epochs=2, total_timesteps=4096, actor_illegal_action_mask=True,
             value_clipping=True, reward_scaling=False, global_gradient_clipping=True, illegal_action_loss_stat="last",
             actor_model_type="DeepMind", actor_activation="relu", lr=1e-3, ent_coef=0.01, clip_eps=0.2, vf_coef=0.5, seed=0)
    c.update(kw)
    return c


@pytest.mark.parametrize("key,value", [("num_envs", 128), ("num_steps", 8), ("minibatch_size", 32), ("update_epochs", 3),
                                       ("total_timesteps", 8192), ("actor_illegal_action_mask", False), ("value_clipping", False),
                                       ("reward_scaling", True), ("global_gradient_clipping", False),
                                       ("illegal_action_loss_stat", "all"), ("actor_model_type", "FAIR"),
                                       ("actor_activation", "tanh"), ("brl_train_tune", 4)])
def test_a_mismatched_shared_key_is_named(key, value):
    from brl_b200.models import make_forward_pass
    from brl_b200.optim import AdamWithClip
    from brl_b200.update import check_population_configs, make_population_update_step
    configs = [_config(), _config(seed=1, lr=3e-4), _config(seed=2, **{key: value})]
    with pytest.raises(ValueError, match=repr(key).replace("[", r"\[")):
        check_population_configs(configs)
    with pytest.raises(ValueError, match=key):
        make_population_update_step(configs, make_forward_pass("relu", "DeepMind", precision="tc"),
                                     [AdamWithClip(1e-3) for _ in configs])


def test_train_population_checks_the_configs_before_any_device_work():
    from brl_b200 import ppo
    with pytest.raises(ValueError, match="minibatch_size"):
        ppo.train_population([_config(), _config(minibatch_size=32)], [0, 1], device="cpu")
    with pytest.raises(ValueError, match="rng"):
        ppo.train_population([_config(), _config()], [0], device="cpu")


def test_everything_else_may_differ_per_learner():
    from brl_b200.update import check_population_configs
    check_population_configs([_config(), _config(seed=7, lr=1e-4, anneal_lr=True, ent_coef=0.0, vf_coef=1.0, clip_eps=0.3,
                                                 max_grad_norm=0.1, gamma=0.9, gae_lambda=0.8, exp_name="b", log_path="/tmp/b")])
    check_population_configs([_config()])
    with pytest.raises(ValueError):
        check_population_configs([])


def test_population_update_step_needs_one_optimizer_per_learner_and_the_tensor_core_net():
    from brl_b200.models import make_forward_pass
    from brl_b200.optim import AdamWithClip
    from brl_b200.update import make_population_update_step
    fp = make_forward_pass("relu", "DeepMind", precision="tc")
    with pytest.raises(ValueError, match="optimizer"):
        make_population_update_step([_config(), _config()], fp, [AdamWithClip(1e-3)])
    with pytest.raises(TypeError):
        make_population_update_step([_config()], object(), [AdamWithClip(1e-3)])


def test_grouped_ops_validate_their_arguments_without_a_gpu():
    from brl_b200 import _lib
    L = _lib.load()
    for name in ("brl_ppo_grad_grouped", "brl_mlp_adam_step_grouped"):  # lazily bound ops: bind them as _lib.call does
        fn, xla = getattr(L, name), getattr(L, name + "_xla")
        fn.restype, fn.argtypes = ctypes.c_int32, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p), ctypes.c_void_p, ctypes.c_size_t]
        xla.restype, xla.argtypes = None, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p), ctypes.c_char_p, ctypes.c_size_t, ctypes.c_void_p]
    sz = L.brl_ppo_grad_grouped_scratch_bytes
    sz.restype, sz.argtypes = ctypes.c_int64, [ctypes.c_int64, ctypes.c_int64]
    stride = L.brl_mlp_param_stride
    stride.restype = ctypes.c_int64
    n = L.brl_mlp_num_params()
    assert stride() >= n and stride() % 64 == 0 and stride() - n < 64
    assert sz(0, 1024) == 0 and sz(3, 0) == 0 and sz(_lib.MAX_LEARNERS + 1, 1024) == 0
    # K learners' minibatch scratches plus the grouped tile counters
    assert sz(1, 1024) > L.brl_mlp_train_scratch_bytes(1024) and sz(3, 1024) > 3 * L.brl_mlp_train_scratch_bytes(1024)
    bufs = (ctypes.c_void_p * 7)()
    gp = _lib.BrlPpoGroupedParams(1024, 3, _lib.PPO_VALUE_CLIPPING, 0, 0)
    assert L.brl_ppo_grad_grouped(None, bufs, ctypes.byref(gp), ctypes.sizeof(gp)) == -2 and b"'traj' is NULL" in L.brl_last_error()
    assert L.brl_ppo_grad_grouped(None, bufs, ctypes.byref(gp), 8) == -1 and b"BrlPpoGroupedParams" in L.brl_last_error()
    gp.n_learners = _lib.MAX_LEARNERS + 1
    assert L.brl_ppo_grad_grouped(None, bufs, ctypes.byref(gp), ctypes.sizeof(gp)) == -1 and b"n_learners" in L.brl_last_error()
    gp.n_learners, gp.batch = 3, -1
    assert L.brl_ppo_grad_grouped(None, bufs, ctypes.byref(gp), ctypes.sizeof(gp)) == -1 and b"batch" in L.brl_last_error()
    # an empty batch is a no-op with NULL buffers (no CUDA call is made)
    for k, b in ((0, 1024), (3, 0)):
        gp.n_learners, gp.batch = k, b
        assert L.brl_ppo_grad_grouped(None, bufs, ctypes.byref(gp), ctypes.sizeof(gp)) == 0
    fake = (ctypes.c_void_p * 7)(*[ctypes.c_void_p(4096)] * 7)
    fake[3] = ctypes.c_void_p(4096 + 8)
    gp.n_learners, gp.batch = 2, 1024
    assert L.brl_ppo_grad_grouped(None, fake, ctypes.byref(gp), ctypes.sizeof(gp)) == -2 and b"'scratch' is not 16-byte" in L.brl_last_error()
    # Adam: opaque = one BrlAdamParams per learner
    ap = (_lib.BrlAdamParams * 2)(_lib.BrlAdamParams(n, 1, 1e-3, 0.9, 0.999, 1e-5, 0.5), _lib.BrlAdamParams(n, 0, 1e-3, 0.9, 0.999, 1e-5, 0.5))
    abufs = (ctypes.c_void_p * 6)()
    assert L.brl_mlp_adam_step_grouped(None, abufs, None, 0) == 0
    assert L.brl_mlp_adam_step_grouped(None, abufs, ctypes.byref(ap), ctypes.sizeof(ap) - 4) == -1 and b"BrlAdamParams" in L.brl_last_error()
    assert L.brl_mlp_adam_step_grouped(None, abufs, ctypes.byref(ap), ctypes.sizeof(ap)) == -2 and b"'params' is NULL" in L.brl_last_error()
    afake = (ctypes.c_void_p * 6)(*[ctypes.c_void_p(4096)] * 6)
    assert L.brl_mlp_adam_step_grouped(None, afake, ctypes.byref(ap), ctypes.sizeof(ap)) == -1 and b"learner 1" in L.brl_last_error()
    many = (_lib.BrlAdamParams * (_lib.MAX_LEARNERS + 1))()
    assert L.brl_mlp_adam_step_grouped(None, afake, ctypes.byref(many), ctypes.sizeof(many)) == -1 and b"at most" in L.brl_last_error()


def test_grouped_ops_are_xla_custom_calls():
    from brl_b200 import _lib
    L = _lib.load()
    assert L.brl_xla_layout(b"brl_ppo_grad_grouped") == b"iiisoos"
    assert L.brl_xla_layout(b"brl_mlp_adam_step_grouped") == b"xixxix"
    for name in ("brl_ppo_grad_grouped", "brl_mlp_adam_step_grouped"):
        assert name in _lib.OPS and name in _lib.LAZY_OPS
        assert hasattr(L, name + "_xla")
