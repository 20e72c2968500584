"""SmartStartContinuous -- drop-in for smartstart/smartexploration/smartexplorationcontinuous.py.

Same constructor kwargs (buffer_size, exploitation_param, exploration_param, eta,
eta_decay_factor, n_ss, print_ss_stuff and every ``nnd_mb_*`` option forwarded 1:1), same
attributes (smart_start_pathing, smart_start_path, eta, nnd_mb_agent, replay_buffer), same
RLAgent methods.  ``get_smart_start_path`` (smartexplorationcontinuous.py:223-305) keeps the
host bookkeeping (candidate sampling, episodic path extraction) and hands the numeric core
-- scipy gaussian_kde fit + evaluate, pseudo-counts, UCB, argmax (:260-280) -- to one CUDA
call, ``Engine.select_start``.
"""
from __future__ import annotations

import time

import numpy as np

from .agents_abstract_classes import ReplayBufferRLAgent, RLAgent
from .nnd_mb_agent import NND_MB_agent
from .numerical import volume_of_n_dimensional_hyperellipsoid
from .replay_buffer import ReplayBuffer


class SmartStartContinuous(RLAgent):
    def __init__(self, agent, env, sess,
                 buffer_size=500000,
                 exploitation_param=1.,
                 exploration_param=2.,
                 eta=0.5,
                 eta_decay_factor=1.,
                 n_ss=1000,
                 print_ss_stuff=True,

                 nnd_mb_final_steps=10,
                 nnd_mb_steps_per_waypoint=1,
                 nnd_mb_mean_per_stepsize=1,
                 nnd_mb_std_per_stepsize=1,
                 nnd_mb_stepsizes_in_waypoint_radii=1,

                 nnd_mb_gamma=.75,
                 nnd_mb_horizontal_penalty_factor=.5,
                 nnd_mb_horizon=20,
                 nnd_mb_num_control_samples=5000,
                 nnd_mb_path_shortcutting=True,
                 nnd_mb_steps_before_giving_up_on_waypoint=5,

                 nnd_mb_save_dir_name="save_untitled",
                 nnd_mb_load_dir_name="untitled_load",
                 nnd_mb_save_training_data=False,
                 nnd_mb_save_resulting_dynamics_model=False,
                 nnd_mb_load_existing_training_data=False,
                 nnd_mb_load_existing_dynamics_model=False,

                 nnd_mb_num_fc_layers=1,
                 nnd_mb_depth_fc_layers=500,
                 nnd_mb_batchsize=512,
                 nnd_mb_lr=0.001,
                 nnd_mb_nEpoch=30,
                 nnd_mb_fraction_use_new=0.9,
                 nnd_mb_num_episodes_for_aggregation=3,
                 nnd_mb_make_aggregated_dataset_noisy=True,
                 nnd_mb_make_training_dataset_noisy=True,
                 nnd_mb_noise_actions_during_MPC_rollouts=True,

                 nnd_mb_verbose=True,

                 nnd_mb_use_threading=True,
                 nnd_mb_num_rollouts_train=25,
                 nnd_mb_num_rollouts_val=20,
                 nnd_mb_dt_steps=3,
                 nnd_mb_steps_per_rollout_train=333,
                 nnd_mb_steps_per_rollout_val=333,

                 *, engine=None, device=0, nnd_mb_extra=None, device_mirror=True, value_net=None,
                 kde_precision="fp32"):
        self.param_dict = {k: v for k, v in locals().items()
                           if k not in ("self", "sess", "env", "agent", "engine", "nnd_mb_extra", "device_mirror", "value_net",
                                        "kde_precision", "__class__")}
        for name in ("self", "sess", "env", "__class__"):
            self.param_dict[name] = "Not serializable"
        self.param_dict["agent"] = agent.get_param_dict()

        self.exploitation_param = exploitation_param
        self.exploration_param = exploration_param
        self.eta = eta
        self.eta_decay_factor = eta_decay_factor
        self.agent = agent
        self.env = env

        if isinstance(agent, ReplayBufferRLAgent) or (
                hasattr(agent, "replay_buffer") and hasattr(agent, "set_replay_buffer_main_agent")):
            self.replay_buffer = agent.replay_buffer
            agent.set_replay_buffer_main_agent(self)
        else:
            self.replay_buffer = ReplayBuffer(self, buffer_size)

        self.n_ss = n_ss
        self.print_ss_stuff = print_ss_stuff
        self.smart_start_pathing = False
        self.smart_start_path = None

        if engine is None:
            from .engine import Engine
            engine = Engine(device)
        self.engine = engine
        # select from the device-resident mirror of the replay buffer's state ring (SURVEY 8f, row f2)
        # whenever the buffer keeps one; False = upload the whole buffer at every selection
        self.device_mirror = bool(device_mirror)
        # SURVEY 8f, row f4: with the critic / actor parameters of the base agent given (the dict
        # Engine.set_value_net takes, or a callable returning it -- called at every selection, so it can
        # export the weights the agent has NOW), V = critic(q, actor(q)) is evaluated on the device in
        # front of the UCB and agent.get_state_value is not called for the candidates
        self.value_net = value_net
        # arithmetic of the selection: "fp32" (default) or "fp64" (scipy's float64 evaluation, Engine.kde_set_precision);
        # set on the engine before every selection, since the engine may be shared
        if kde_precision not in ("fp32", "fp64"):
            raise ValueError("kde_precision must be 'fp32' or 'fp64', got %r" % (kde_precision,))
        self.kde_precision = kde_precision

        self.nnd_mb_agent = NND_MB_agent(
            env, sess, replay_buffer=self.replay_buffer,
            final_steps=nnd_mb_final_steps, steps_per_waypoint=nnd_mb_steps_per_waypoint,
            mean_per_stepsize=nnd_mb_mean_per_stepsize, std_per_stepsize=nnd_mb_std_per_stepsize,
            stepsizes_in_waypoint_radii=nnd_mb_stepsizes_in_waypoint_radii,
            gamma=nnd_mb_gamma, horizontal_penalty_factor=nnd_mb_horizontal_penalty_factor,
            horizon=nnd_mb_horizon, num_control_samples=nnd_mb_num_control_samples,
            path_shortcutting=nnd_mb_path_shortcutting,
            steps_before_giving_up_on_waypoint=nnd_mb_steps_before_giving_up_on_waypoint,
            save_dir_name=nnd_mb_save_dir_name, load_dir_name=nnd_mb_load_dir_name,
            save_training_data=nnd_mb_save_training_data,
            save_resulting_dynamics_model=nnd_mb_save_resulting_dynamics_model,
            load_existing_training_data=nnd_mb_load_existing_training_data,
            load_existing_dynamics_model=nnd_mb_load_existing_dynamics_model,
            num_fc_layers=nnd_mb_num_fc_layers, depth_fc_layers=nnd_mb_depth_fc_layers,
            batchsize=nnd_mb_batchsize, lr=nnd_mb_lr, nEpoch=nnd_mb_nEpoch,
            fraction_use_new=nnd_mb_fraction_use_new,
            num_episodes_for_aggregation=nnd_mb_num_episodes_for_aggregation,
            make_aggregated_dataset_noisy=nnd_mb_make_aggregated_dataset_noisy,
            make_training_dataset_noisy=nnd_mb_make_training_dataset_noisy,
            noise_actions_during_MPC_rollouts=nnd_mb_noise_actions_during_MPC_rollouts,
            verbose=nnd_mb_verbose, use_threading=nnd_mb_use_threading,
            num_rollouts_train=nnd_mb_num_rollouts_train, num_rollouts_val=nnd_mb_num_rollouts_val,
            dt_steps=nnd_mb_dt_steps, steps_per_rollout_train=nnd_mb_steps_per_rollout_train,
            steps_per_rollout_val=nnd_mb_steps_per_rollout_val,
            engine=engine, **(nnd_mb_extra or {}))
        self.times_for_smart_start = []
        self.last_selection = None      # (buffer index, ucb) of the latest choice, for inspection

    def get_param_dict(self):
        return self.param_dict

    def get_summary_name(self):
        base = self.agent.get_summary_name() if hasattr(self.agent, "get_summary_name") \
            else self.agent.__class__.__name__
        return "SmartStartC_" + base

    @property
    def normal_agent_pathing(self):
        return not self.smart_start_pathing

    def reduce_eta(self):
        self.eta = self.eta * self.eta_decay_factor

    # ------------------------------------------------------------------ stage 1
    def _candidate_states(self, indices):
        rb = self.replay_buffer
        if hasattr(rb, "states_s2"):
            return np.asarray(rb.states_s2(indices), dtype=np.float64)
        return np.asarray([np.asarray(rb.buffer[int(i)][4], dtype=np.float64) for i in indices])

    def get_smart_start_path(self):
        """UCB1 choice of the smart-start state; returns the stored path leading to it (list of
        states, last one = the smart start) or None when there is nothing to choose from."""
        if len(self.replay_buffer) == 0:
            return None
        possible_start_indices = self.replay_buffer.get_possible_smart_start_indices(self.n_ss)
        if possible_start_indices is None:
            return None
        if self.nnd_mb_agent.radii is not None:
            one_radii_volume = volume_of_n_dimensional_hyperellipsoid(self.nnd_mb_agent.radii)
        else:
            one_radii_volume = 1
        self.engine.kde_set_precision(self.kde_precision)
        ring = self.replay_buffer.state_ring() if hasattr(self.replay_buffer, "state_ring") else None
        mirror = ring is not None and self.device_mirror
        values = None
        if self.value_net is not None:
            net = self.value_net() if callable(self.value_net) else self.value_net
            if net is not getattr(self, "_value_net_on_device", None):
                self.engine.set_value_net(net)
                self._value_net_on_device = net
        if self.value_net is None or not mirror:
            possible_ss_states = self._candidate_states(possible_start_indices)
        if self.value_net is None:
            values = np.asarray(self.agent.get_state_value(possible_ss_states)).T.reshape(-1)   # 1 x m
        if mirror:
            # the buffer's states already live on the device (incremental mirror): only the m candidate
            # indices (and the values, unless the device computes them) are uploaded
            best_j, best_ucb, _, _ = self.engine.select_start_mirror(
                ring, possible_start_indices, values, len(self.replay_buffer),
                one_radii_volume, self.exploitation_param, self.exploration_param)
        else:
            all_states = np.asarray(self.replay_buffer.get_all_states(), dtype=np.float64)
            if all_states.ndim == 1:
                all_states = all_states[:, None]
            best_j, best_ucb, _, _ = self.engine.select_start(
                all_states, possible_ss_states, values, len(self.replay_buffer),
                one_radii_volume, self.exploitation_param, self.exploration_param)
        smart_start_index = int(possible_start_indices[best_j])
        self.last_selection = (smart_start_index, best_ucb)
        return self.replay_buffer.get_episodic_path_to_buffer_index(smart_start_index)

    # ------------------------------------------------------------------ RLAgent API
    def get_action(self, state):
        if self.smart_start_pathing:
            return self.nnd_mb_agent.get_action(state)
        return self.agent.get_action(state)

    def observe(self, state, action, reward, new_state, done):
        self.replay_buffer.add(self, state, action, reward, done, new_state)
        self.agent.observe(state, action, reward, new_state, done)
        if self.smart_start_pathing:
            self.nnd_mb_agent.observe(state, action, reward, new_state, done)
            if self.nnd_mb_agent.close_enough_to_goal(new_state):
                self.smart_start_pathing = False
                if self.print_ss_stuff:
                    print("distance to goal: " + str(
                        self.nnd_mb_agent.distance_function(new_state, self.smart_start_path[-1])))
                    print("END OF SMART START STUFFS")

    def start_new_episode(self, state):
        self.smart_start_pathing = False
        self.smart_start_path = None
        if np.random.rand() <= self.eta:
            t0 = time.time()
            self.smart_start_path = self.get_smart_start_path()
            elapsed = time.time() - t0
            if self.smart_start_path:
                self.times_for_smart_start.append(elapsed)
                if self.print_ss_stuff:
                    print("Calculate Smart Start Path Time: " + str(elapsed), end='')
                    print("\npath exists")
                self.nnd_mb_agent.start_new_episode_plan(state, self.smart_start_path)
                if not self.nnd_mb_agent.close_enough_to_goal(state):
                    self.smart_start_pathing = True
                    if self.print_ss_stuff:
                        print("SMART_START START!!!")
        self.agent.start_new_episode(state)
        self.replay_buffer.start_new_episode(self)

    def end_episode(self):
        self.reduce_eta()
        self.agent.end_episode()
        self.smart_start_pathing = False
        self.smart_start_path = None

    def render(self, env, **kwargs):
        return env.render()
