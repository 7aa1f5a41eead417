"""GPU: the reference's UNMODIFIED PPO2 learner consumes the engine's env unchanged (BASELINE.json north_star: "the existing
algorithm/ PPO2 ... loops consume it unchanged").

The collection loop and the learner of demonstration/PPO2/PPO2-4-CartPoleAngleOnly/train.py (:138-222) -- reference
``Proximal_Policy_Optimization2``, ``PPOActor_Gaussian`` / ``PPOCritic``, ``Normalization``, seed 3407 -- are run twice with the
same loop body: once on the reference's own env, once on ``rlp.single(rlp.CartPoleAngleOnly(variant='ppo2'))``.  The only
difference is where ``reset(True)`` takes its initial condition from: the reference draws from the global numpy stream, which
no per-instance generator reproduces, so the engine run replays the initial conditions the reference run drew (a wrapper
around ``reset``; the loop itself is untouched).  Same torch seed => same exploration noise, so identical environments give
identical rollouts and identical parameters after ``agent.learn()``.

The reference comes from /root/reference in the build container and from the byte-compiled staging oracle/_ref/ on the GPU
box (oracle/stage_reference.py; checker only)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _load():
    from oracle import ref_shim as R
    if not R.available():
        pytest.skip("runs the original project's own PPO2 learner code, which is not part of the repository: "
                    "no reference tree (RLP_REFERENCE, or oracle/_ref staged by build())")
    R.install()
    with R.quiet():
        envmod = R.load_file("demonstration/PPO2/PPO2-4-CartPoleAngleOnly/cartpole_angleonly.py", "ref_learner_env")
        cls = R.load("utils.classes")
        ppo = R.load("algorithm.policy_base.Proximal_Policy_Optimization2")
    return R, envmod, cls, ppo


def _agent(env, cls, ppo, buffer_size):
    env_msg = {'state_dim': env.state_dim, 'action_dim': env.action_dim, 'name': env.name, 'action_range': env.action_range}
    ppo_msg = {'gamma': 0.999, 'K_epochs': 5, 'eps_clip': 0.2, 'buffer_size': buffer_size, 'state_dim': env.state_dim,
               'action_dim': env.action_dim, 'a_lr': 3e-4, 'c_lr': 1e-3, 'set_adam_eps': True, 'lmd': 0.95,
               'use_adv_norm': True, 'mini_batch_size': 64, 'entropy_coef': 0.01, 'use_grad_clip': True,
               'use_lr_decay': True, 'max_train_steps': int(5e6), 'using_mini_batch': False}   # train.py:141-158
    ar = np.array(env.action_range)
    return ppo.Proximal_Policy_Optimization2(
        env_msg=env_msg, ppo_msg=ppo_msg,
        actor=cls.PPOActor_Gaussian(state_dim=env.state_dim, action_dim=env.action_dim, a_min=ar[:, 0], a_max=ar[:, 1],
                                    init_std=env.fm / 3, use_orthogonal_init=True),
        critic=cls.PPOCritic(state_dim=env.state_dim, use_orthogonal_init=True))


def _train(R, env, agent, reward_norm, epochs):
    """train.py:184-222, verbatim loop body; returns the rollouts and the parameters after every learn()."""
    rollouts, params, total = [], [], 0
    env.is_terminal = True
    for _ in range(epochs):
        idx, rows = 0, []
        with R.quiet():
            while idx < agent.buffer.batch_size:
                if env.is_terminal:
                    env.reset(True)
                else:
                    env.current_state = env.next_state.copy()
                    a, a_lp = agent.choose_action(env.current_state)
                    env.step_update(a)
                    success = 1 if (env.is_terminal and env.terminal_flag != 3) else 0
                    agent.buffer.append(s=env.current_state, a=a, log_prob=a_lp, r=reward_norm(env.reward),
                                        s_=env.next_state, done=1.0 if env.is_terminal else 0.0, success=success, index=idx)
                    rows.append(np.concatenate([env.current_state, np.ravel(a), env.next_state,
                                                [env.reward, float(env.is_terminal), float(env.terminal_flag)]]))
                    idx += 1
            total += idx
            agent.learn(total, buf_num=1)
        rollouts.append(np.array(rows))
        params.append(np.concatenate([p.detach().cpu().numpy().ravel()
                                      for net in (agent.actor, agent.critic) for p in net.parameters()]))
    return rollouts, params


def test_reference_ppo2_learner_on_engine_env_matches_reference_env():
    import torch
    import reinforcementlearningplatform_b200 as rlp
    R, envmod, cls, ppo = _load()
    T, epochs = 400, 2

    # ---- run A: reference env; every reset's initial condition is recorded
    np.random.seed(3407)
    torch.manual_seed(3407)
    with R.quiet():
        ref_env = envmod.CartPoleAngleOnly(0.)
    inits = []
    ref_reset = ref_env.reset

    def recording_reset(random=True):
        ref_reset(random)
        inits.append((np.array([ref_env.theta, ref_env.dtheta, ref_env.x, ref_env.dx], dtype=float), float(ref_env.time)))
    ref_env.reset = recording_reset
    roll_a, par_a = _train(R, ref_env, _agent(ref_env, cls, ppo, T), cls.Normalization(shape=1), epochs)

    # ---- run B: the engine's env behind the rl_base view, same loop, initial conditions replayed
    np.random.seed(3407)
    torch.manual_seed(3407)
    eng = rlp.single(rlp.CartPoleAngleOnly(n_envs=1, variant='ppo2'))
    assert eng.state_dim == ref_env.state_dim and eng.action_dim == ref_env.action_dim
    assert np.array_equal(np.asarray(eng.action_range, dtype=float), np.asarray(ref_env.action_range, dtype=float))
    assert eng.fm == ref_env.fm              # PPOActor_Gaussian(init_std=env.fm / 3)
    replay = iter(inits)
    eng_reset = eng.reset

    def replaying_reset(random=True):
        eng_reset(random)
        state, time0 = next(replay)
        eng.set_state(state, time0)
    eng.reset = replaying_reset
    roll_b, par_b = _train(R, eng, _agent(eng, cls, ppo, T), cls.Normalization(shape=1), epochs)

    # ---- identical rollouts (states, actions, rewards, flags) and identical parameters after each update
    for e in range(epochs):
        a, b = roll_a[e], roll_b[e]
        assert a.shape == b.shape == (T, a.shape[1])
        assert np.array_equal(a[:, -2:], b[:, -2:]), "is_terminal / terminal_flag differ"
        err = np.max(np.abs(a - b) / np.maximum(1.0, np.abs(a)))
        assert err <= 1e-12, (e, err)
        perr = np.max(np.abs(par_a[e] - par_b[e]))
        assert perr <= 1e-6, (e, perr)
    assert next(replay, None) is None       # both runs went through the same number of episodes


def _train_uav(R, env, agent, reward_norm, epochs, reset_fn):
    """PPO2-4-UavFntsmcParamPos/train.py:273-313, verbatim loop body (three-call protocol, state normalisers of the env)."""
    rollouts, params, total = [], [], 0
    env.is_terminal = True
    for _ in range(epochs):
        idx, rows = 0, []
        with R.quiet():
            while idx < agent.buffer.batch_size:
                if env.is_terminal:
                    reset_fn()
                else:
                    env.current_state = env.next_state.copy()
                    s = env.current_state_norm(env.current_state, update=True)
                    a, a_log_prob = agent.choose_action(s)
                    new_SMC_param = a.copy()
                    env.get_param_from_actor(new_SMC_param)
                    action_4_uav = env.generate_action_4_uav()
                    env.step_update(action_4_uav)
                    success = 1.0 if (env.is_terminal and (env.terminal_flag != 1)) else 0.
                    agent.buffer.append(s=s, a=a, log_prob=a_log_prob, r=reward_norm(env.reward),
                                        s_=env.next_state_norm(env.next_state, update=True),
                                        done=1.0 if env.is_terminal else 0.0, success=success, index=idx)
                    rows.append(np.concatenate([env.current_state, np.ravel(a), env.next_state, np.ravel(s),
                                                [env.reward, float(env.is_terminal), float(env.terminal_flag)]]))
                    idx += 1
            total += idx
            agent.learn(total, buf_num=1)
        rollouts.append(np.array(rows))
        params.append(np.concatenate([p.detach().cpu().numpy().ravel()
                                      for net in (agent.actor, agent.critic) for p in net.parameters()]))
    return rollouts, params


def _uav_agent(env, cls, ppo, buffer_size):
    env_msg = {'state_dim': env.state_dim, 'action_dim': env.action_dim, 'name': env.name, 'action_range': env.action_range}
    ppo_msg = {'gamma': 0.99, 'K_epochs': 5, 'eps_clip': 0.2, 'buffer_size': buffer_size, 'state_dim': env.state_dim,
               'action_dim': env.action_dim, 'a_lr': 1e-4, 'c_lr': 1e-3, 'set_adam_eps': True, 'lmd': 0.95,
               'use_adv_norm': True, 'mini_batch_size': 64, 'entropy_coef': 0.01, 'use_grad_clip': True,
               'use_lr_decay': True, 'max_train_steps': int(5e6), 'using_mini_batch': False}   # train.py:224-240
    ar = np.array(env.action_range)
    return ppo.Proximal_Policy_Optimization2(
        env_msg=env_msg, ppo_msg=ppo_msg,
        actor=cls.PPOActor_Gaussian(state_dim=env.state_dim, action_dim=env.action_dim, a_min=ar[:, 0], a_max=ar[:, 1],
                                    init_std=0.4, use_orthogonal_init=True),
        critic=cls.PPOCritic(state_dim=env.state_dim, use_orthogonal_init=True))


def test_reference_ppo2_learner_on_engine_uav_pos_env_matches_reference_env():
    """The headline env: uav_pos_ctrl_RL under the reference learner, get_param_from_actor / generate_action_4_uav /
    step_update and the env's own current_state_norm / next_state_norm as train.py calls them."""
    import torch
    import reinforcementlearningplatform_b200 as rlp
    from helpers import env_specs
    from oracle import ref_adapters as A
    from reinforcementlearningplatform_b200.envs import uav as U
    R, _, cls, ppo = _load()
    T, epochs = 300, 2

    ad = A.REGISTRY["uav_pos"][0]()
    np.random.seed(3407)
    torch.manual_seed(3407)
    with R.quiet():
        ref_env = ad.make()
    inits = []

    def ref_reset():
        ad.reset(ref_env)                                   # reset_pos_ctrl_param('zero') + reset_uav_pos_ctrl_RL_tracking
        inits.append(ad.internal(ref_env))
    roll_a, par_a = _train_uav(R, ref_env, _uav_agent(ref_env, cls, ppo, T), cls.Normalization(shape=1), epochs, ref_reset)

    np.random.seed(3407)
    torch.manual_seed(3407)
    ecls, kw = env_specs()["uav_pos"]
    eng = rlp.single(ecls(n_envs=1, **kw))
    assert eng.state_dim == ref_env.state_dim and eng.action_dim == ref_env.action_dim
    assert np.array_equal(np.asarray(eng.action_range, dtype=float), np.asarray(ref_env.action_range, dtype=float))
    replay = iter(inits)
    zero = U.train_pos_ctrl_param()
    for name in ("k1", "k2", "gamma", "lmd"):
        setattr(zero, name, 0.01 * np.ones(3))

    def eng_reset():
        eng.reset_uav_pos_ctrl_RL_tracking(random_trajectroy=True, random_pos0=False, new_att_ctrl_param=None,
                                           new_pos_ctrl_parma=zero, outer_param=None)
        state, time0 = next(replay)
        eng.set_state(state, time0)
    roll_b, par_b = _train_uav(R, eng, _uav_agent(eng, cls, ppo, T), cls.Normalization(shape=1), epochs, eng_reset)

    worst, pworst = 0.0, 0.0
    for e in range(epochs):
        a, b = roll_a[e], roll_b[e]
        assert a.shape == b.shape and a.shape[0] == T
        assert np.array_equal(a[:, -2:], b[:, -2:]), "is_terminal / terminal_flag differ"
        worst = max(worst, float(np.max(np.abs(a - b) / np.maximum(1.0, np.abs(a)))))
        pworst = max(pworst, float(np.max(np.abs(par_a[e] - par_b[e]))))
    print(f"uav_pos under the reference learner: rollout mixed error {worst:.3e}, parameter error {pworst:.3e}, "
          f"{len(inits)} episodes")
    # measured on B200: 5.9e-14 over the two 300-step buffers, parameters bit-equal after both updates
    assert worst <= 1e-12, worst
    assert pworst <= 1e-7, pworst
    assert next(replay, None) is None
