"""NND_MB_agent -- MPC navigator; drop-in for smartstart/RLAgents/NND_MB_agent.py.

Constructor kwargs, attributes read from outside (radii, distance_function, path_to_follow,
desired_states, current_desired_state(_index), distances_left; rlTrain.py:173,209,234-251)
and method names are the reference's.  What changed underneath:

  get_best_sim_actions (NND_MB_agent.py:498-520): one call into the CUDA engine
      (sample -> H-step MLP rollout -> trajectory scoring -> arg-max, all on the GPU)
      instead of H sess.run round trips + ~25 numpy passes per step.
  start_new_episode_plan (:375-423): same host geometry (numerical.py), then the plan
      (desired_states, distances_left, radii) is uploaded once with Engine.set_plan.
  train_dynamics_model (:437-480): torch Adam loop (dynamics_model.py), weights re-uploaded.

Extra keyword-only options (all default to the reference behaviour):
  engine / device     share an Engine or create one on cuda:<device>
  penalty_mode        "reference" (global projection coefficient, Q1) | "per_sample"
  precision           "auto" | "fp32" | "bf16_tc" | "fp64"; "fp64" rolls out and scores in float64 like the
                      reference (its decision up to the summation order of the GEMMs and reductions, also
                      when the best two scores are closer than the FP32 / BF16 tolerances), several times
                      slower than "bf16_tc"; "auto" never picks it
  train_precision     "fp32" | "fp64"; arithmetic of the device trainer behind train_dynamics_model.  "fp64"
                      trains in float64 like the reference's graph, so a retrained model stays the reference's
                      up to the summation order of the GEMMs; the reference-faithful configuration is
                      precision="fp64", train_precision="fp64"
  device_sampling     False: the actions of numpy.random.uniform exactly like :500-501 -- the global
                      MT19937 stream, generated on the GPU from np.random.get_state() and advanced with
                      set_state (host_rng=True draws them on the host and uploads them instead, False
                      always uses the GPU; the default None draws batches of up to HOST_DRAW_MAX samples
                      on the host, where that is faster -- the numbers are the same either way);
                      True: Philox on the GPU (a different, shard-invariant stream)
  planner             a distributed.ShardedPlanner: the K sequences of every decision are sharded
                      over the ranks of its torch.distributed group (all ranks run the agent in
                      lock-step with identical numpy seeds; every rank generates its own slice of the
                      one global draw, so the sharded decision equals the single-GPU one; with
                      host_rng=True every rank draws only its own K/world sequences)
"""
from __future__ import annotations

import os

import numpy as np
import numpy.random as npr

from .agents_abstract_classes import NavigationRLAgent
from .dynamics_model import Dyn_Model
from .numerical import (elliptical_euclidean_distance_function_generator,
                        get_start_waypoints_final_states_steps, path_deltas_stds_and_means_per_dim,
                        path_shortcutter, radii_calc)
from .replay_buffer import ReplayBuffer


def plan_from_path(path_to_follow, *, mean_per_stepsize, std_per_stepsize, stepsizes_in_waypoint_radii,
                   path_shortcutting, theta, steps_per_waypoint, engine=None):
    """Host part of start_new_episode_plan (NND_MB_agent.py:385-418): radii from the step-size
    statistics, elliptical distance, optional shortcutting, waypoints, distances left."""
    stds, means = path_deltas_stds_and_means_per_dim(path_to_follow)
    radii = radii_calc(means, stds, mean_per_stepsize, std_per_stepsize, stepsizes_in_waypoint_radii)
    dist = elliptical_euclidean_distance_function_generator(radii)
    followed = path_shortcutter(path_to_follow, dist, theta, engine=engine) if path_shortcutting else path_to_follow
    desired = np.asarray(get_start_waypoints_final_states_steps(followed, steps_per_waypoint))
    if len(desired) >= 2:
        hops = np.append(dist(desired[:-1], desired[1:]), 0.0)
        # distances_left[i] = sum(hops[i:]) accumulated front to back like the reference's sum()
        left = np.asarray([sum(hops[i:].tolist()) for i in range(len(desired))])
    else:
        left = np.asarray([0])
    return dict(stds=stds, radii=radii, distance_function=dist, path_to_follow=followed,
                desired_states=desired, distances_left=left)


def _collect_random_rollouts(env, num_rollouts, steps_per_rollout):
    """Random-policy data collection (stands in for perform_rollouts / CollectSamples,
    NND_MB_agent.py:236-246): returns (states [R][T+1, d], controls [R][T, da])."""
    low, high = np.asarray(env.action_space.low, dtype=np.float64), np.asarray(env.action_space.high, dtype=np.float64)
    all_s, all_a = [], []
    for _ in range(num_rollouts):
        obs = np.asarray(env.reset(), dtype=np.float64)
        ss, aa = [obs], []
        for _ in range(steps_per_rollout):
            a = npr.uniform(low, high)
            out = env.step(a)
            obs, done = np.asarray(out[0], dtype=np.float64), bool(out[2])
            ss.append(obs)
            aa.append(np.asarray(a, dtype=np.float64).reshape(-1))
            if done:
                break
        all_s.append(np.array(ss))
        all_a.append(np.array(aa))
    return all_s, all_a


class NND_MB_agent(NavigationRLAgent):
    model_subdirectory_name = "NND_MB_agent"
    tf_datatype = "float64"
    noiseToSignal = 0.01
    actions_ag = 'nc'
    HOST_DRAW_MAX = 4096        # K*H*da up to which the host draws the action samples itself (host_rng=None)

    def __init__(self, env, sess,

                 replay_buffer=None, BUFFER_SIZE=10000,

                 final_steps=10, steps_per_waypoint=1, mean_per_stepsize=1, std_per_stepsize=1,
                 stepsizes_in_waypoint_radii=1,

                 gamma=.75, horizontal_penalty_factor=.5, horizon=20, num_control_samples=5000,
                 path_shortcutting=True, steps_before_giving_up_on_waypoint=5,

                 save_dir_name="save_untitled", load_dir_name="untitled_load",
                 save_training_data=False, save_resulting_dynamics_model=False,
                 load_existing_training_data=False, load_existing_dynamics_model=False,

                 num_fc_layers=1, depth_fc_layers=500, batchsize=512, lr=0.001, nEpoch=30,
                 fraction_use_new=0.9, num_episodes_for_aggregation=3,
                 make_aggregated_dataset_noisy=True, make_training_dataset_noisy=True,
                 noise_actions_during_MPC_rollouts=True,

                 verbose=True,

                 use_threading=True, num_rollouts_train=25, num_rollouts_val=20, dt_steps=3,
                 steps_per_rollout_train=333, steps_per_rollout_val=333,

                 *, engine=None, device=0, penalty_mode="reference", precision="auto",
                 device_sampling=False, host_rng=None, training_data=None, model_root=None, seed=None,
                 planner=None, train_precision="fp32"):
        self.theta = 1            # distance function is scaled instead (NND_MB_agent.py:135-138)
        self.final_steps = final_steps
        self.gamma = gamma
        self.horizontal_penalty_factor = horizontal_penalty_factor
        self.env = env
        self.N = num_control_samples
        self.horizon = horizon
        self.steps_per_waypoint = steps_per_waypoint
        self.mean_per_stepsize = mean_per_stepsize
        self.std_per_stepsize = std_per_stepsize
        self.stepsizes_in_waypoint_radii = stepsizes_in_waypoint_radii
        self.use_existing_dynamics_model = load_existing_dynamics_model
        self.make_aggregated_dataset_noisy = make_aggregated_dataset_noisy
        self.nEpochs = nEpoch
        self.fraction_use_new = fraction_use_new
        self.num_episodes_for_aggregation = num_episodes_for_aggregation
        self.path_shortcutting = path_shortcutting
        self.steps_before_giving_up_on_waypoint = steps_before_giving_up_on_waypoint
        self.num_episodes_finished = 0
        self.actions_done_for_current_waypoint = None
        self.radii = None
        self.distance_function = None
        self.stds = None
        self.path_to_follow = None
        self.desired_states = None
        self.current_desired_state_index = None
        self.distances_left = None
        self.save_resulting_dynamics_model = save_resulting_dynamics_model
        self.noise_amount = 0.005 if noise_actions_during_MPC_rollouts else 0
        self.sess = sess
        self.verbose = verbose
        self.penalty_mode = penalty_mode
        self.precision = precision
        self.device_sampling = device_sampling
        self.host_rng = host_rng
        self.planner = planner
        self._plan_calls = 0

        root = model_root or os.path.join(os.getcwd(), "models")
        self.load_dir = os.path.join(root, self.model_subdirectory_name, load_dir_name)
        self.save_dir = os.path.join(root, self.model_subdirectory_name, save_dir_name) \
            if (save_resulting_dynamics_model or save_training_data) else None

        if engine is None:
            from .engine import Engine
            engine = Engine(device)
        self.engine = engine

        self.replay_buffer = replay_buffer if replay_buffer is not None else ReplayBuffer(self, BUFFER_SIZE)

        # ---- initial training data (NND_MB_agent.py:208-296)
        if training_data is not None:
            self.dataX, self.dataY, self.dataZ = (np.array(training_data[k], dtype=np.float64)
                                                  for k in ("dataX", "dataY", "dataZ"))
            self.states_val = training_data.get("states_val")
            self.controls_val = training_data.get("controls_val")
        elif load_existing_training_data:
            td = os.path.join(self.load_dir, "training_data")
            self.dataX = np.load(os.path.join(td, "dataX.npy"))
            self.dataY = np.load(os.path.join(td, "dataY.npy"))
            self.dataZ = np.load(os.path.join(td, "dataZ.npy"))
            self.states_val = np.load(os.path.join(td, "states_val.npy"))
            self.controls_val = np.load(os.path.join(td, "controls_val.npy"))
        else:
            if verbose:
                print("Performing rollouts to collect training data")
            states, controls = _collect_random_rollouts(env, num_rollouts_train, steps_per_rollout_train)
            self.states_val, self.controls_val = _collect_random_rollouts(env, num_rollouts_val,
                                                                          steps_per_rollout_val)
            self.dataX = np.concatenate([s[:-1] for s in states])
            self.dataY = np.concatenate(controls)
            self.dataZ = np.concatenate([s[1:] - s[:-1] for s in states])
            if make_training_dataset_noisy:
                self.dataX = self._add_noise(self.dataX)
                self.dataZ = self._add_noise(self.dataZ)
            if save_training_data:
                td = os.path.join(self.save_dir, "training_data")
                os.makedirs(td, exist_ok=True)
                for nm in ("dataX", "dataY", "dataZ"):
                    np.save(os.path.join(td, nm + ".npy"), getattr(self, nm))

        # ---- normalisation: every component mean 0 / std 1 (:302-315)
        with np.errstate(divide="ignore", invalid="ignore"):
            self.mean_x = np.mean(self.dataX, axis=0)
            self.dataX = self.dataX - self.mean_x
            self.std_x = np.std(self.dataX, axis=0)
            self.dataX = np.nan_to_num(self.dataX / self.std_x)
            self.mean_y = np.mean(self.dataY, axis=0)
            self.dataY = self.dataY - self.mean_y
            self.std_y = np.std(self.dataY, axis=0)
            self.dataY = np.nan_to_num(self.dataY / self.std_y)
            self.mean_z = np.mean(self.dataZ, axis=0)
            self.dataZ = self.dataZ - self.mean_z
            self.std_z = np.std(self.dataZ, axis=0)
            self.dataZ = np.nan_to_num(self.dataZ / self.std_z)
        self.inputs = np.concatenate((self.dataX, self.dataY), axis=1)
        self.outputs = np.copy(self.dataZ)
        assert self.inputs.shape[0] == self.outputs.shape[0]

        self.dyn_model = Dyn_Model(self.inputs.shape[1], self.outputs.shape[1], self.sess, lr, batchsize,
                                   num_fc_layers, depth_fc_layers, self.mean_x, self.mean_y, self.mean_z,
                                   self.std_x, self.std_y, self.std_z, self.tf_datatype, verbose,
                                   engine=self.engine, seed=seed, precision=train_precision)
        self.dyn_model.push_to_engine()
        # the default decision path draws numpy's stream on the GPU: build its jump-ahead plan now, not in the
        # first decision
        try:
            da = int(np.prod(env.action_space.shape))
            n_total = self.N * self.horizon * da
            if not device_sampling and host_rng is not True and n_total > self.HOST_DRAW_MAX:
                first, count = 0, n_total
                if planner is not None:
                    from .distributed import shard_bounds
                    k0, kl = shard_bounds(self.N, planner.world, planner.rank)
                    first, count = k0 * self.horizon * da, kl * self.horizon * da
                self.engine.mt19937_warm(n_total, np.asarray(env.action_space.low, dtype=np.float64).reshape(-1),
                                         np.asarray(env.action_space.high, dtype=np.float64).reshape(-1), first, count)
        except AttributeError:
            pass            # an environment without a Box-like action space: nothing to prepare

    def _add_noise(self, data):
        """helper_funcs.add_noise (helper_funcs.py:10-16): per-column gaussian noise with
        std = noiseToSignal * column mean; columns whose mean is <= 0 stay clean (reference quirk)."""
        out = np.array(data, dtype=np.float64)
        scale = self.noiseToSignal * out.mean(axis=0)
        for j in range(out.shape[1]):
            if scale[j] > 0:
                out[:, j] += npr.normal(0, abs(scale[j]), (out.shape[0],))
        return out

    def get_param_dict(self):
        return None

    # ------------------------------------------------------------------ acting
    def get_action(self, state):
        return self.get_action_with_predicted_states(state)[0]

    def get_action_with_predicted_states(self, state):
        self.actions_done_for_current_waypoint += 1
        best_action, _, _, best_path = self.get_best_sim_actions(state)
        action_to_take = np.copy(best_action)
        if self.actions_ag in ('nn', 'nc'):                         # executed action is noisy
            action_to_take = action_to_take + self.noise_amount * npr.normal(size=action_to_take.shape)
        return action_to_take, best_path

    def get_best_sim_actions(self, curr_nn_state):
        """(best_action [da], best_sim_number, best_sequence [H, da], best_path [H+1, d])."""
        space = self.env.action_space
        cached = getattr(self, "_bounds_cache", None)
        if cached is None or cached[0] is not space.low or cached[1] is not space.high:
            # contiguous float64 copies of the bounds, redone only when the environment hands out new arrays
            cached = (space.low, space.high, np.ascontiguousarray(space.low, dtype=np.float64).reshape(-1),
                      np.ascontiguousarray(space.high, dtype=np.float64).reshape(-1), int(np.prod(space.shape)))
            self._bounds_cache = cached
        low, high, da = cached[2], cached[3], cached[4]
        common = dict(gamma=self.gamma, horizontal_penalty_factor=self.horizontal_penalty_factor,
                      penalty_mode=self.penalty_mode, precision=self.precision)
        K_draw, plan = self.N, self.engine.plan
        if self.planner is not None:
            from .distributed import shard_bounds
            K_draw = shard_bounds(self.N, self.planner.world, self.planner.rank)[1]
            plan = self.planner.plan
        if self.device_sampling:
            self._plan_calls += 1
            seed = int(npr.randint(0, 2 ** 31 - 1)) * 4099 + self._plan_calls
            res = plan(curr_nn_state, self.current_desired_state_index, K=self.N,
                       H=self.horizon, seed=seed, act_low=low, act_high=high, **common)
        elif self.host_rng is False or (self.host_rng is None and self.N * self.horizon * da > self.HOST_DRAW_MAX):
            # npr.uniform(low, high, (N, H, da)) of :500-501, bit for bit, but generated on the GPU from
            # numpy's own generator state (MT19937 jump-ahead, csrc/mt19937.cu): the global stream
            # advances exactly as if the host had drawn, no K*H*da host RNG and no upload.  A sharded
            # planner generates each rank's slice of the SAME draw.
            # (the library reads and advances numpy's state struct in place when it can be reached:
            # np.random.get_state() + set_state() cost 50-150 us per decision)
            addr = self.engine.global_rng_address()
            res = plan(curr_nn_state, self.current_desired_state_index, K=self.N, H=self.horizon,
                       act_low=low, act_high=high, rng_state=addr if addr is not None else npr.get_state(), **common)
            if addr is None:
                npr.set_state(res["rng_state"])
        else:
            # the same draw on the host (legacy uniform = low + (high - low) * random_sample in draw
            # order, without npr.uniform's slow broadcast path).  host_rng=True under a sharded planner:
            # every rank draws only its own K/world sequences (a different, cheaper draw); the automatic
            # choice for small batches draws the whole array so that the decision does not depend on it
            local_only = self.planner is not None and self.host_rng is True
            all_samples = npr.random_sample((K_draw if local_only else self.N, self.horizon, da))
            all_samples *= np.asarray(high, dtype=np.float64) - np.asarray(low, dtype=np.float64)
            all_samples += np.asarray(low, dtype=np.float64)
            if self.planner is not None:
                key = "local_actions" if local_only else "actions"
                res = plan(curr_nn_state, self.current_desired_state_index, K=self.N, H=self.horizon,
                           **{key: all_samples}, **common)
            else:
                res = plan(curr_nn_state, self.current_desired_state_index, actions=all_samples, **common)
        best_sequence = res["best_sequence"]
        return np.copy(best_sequence[0]), res["best_k"], best_sequence, res["best_path"]

    def observe(self, state, action, reward, new_state, done):
        self.replay_buffer.add(self, state, action, reward, done, new_state)
        d_cur = self.distance_function(new_state, self.current_desired_state)
        d_next = self.distance_function(new_state, self.next_desired_state)
        stuck = (self.actions_done_for_current_waypoint > self.steps_before_giving_up_on_waypoint and
                 self.current_desired_state_index != len(self.desired_states) - 1)
        if self.move_to_next(new_state, self.current_desired_state_index, d_cur, d_next) or stuck:
            self.current_desired_state_index += 1
            self.actions_done_for_current_waypoint = 0

    def start_new_episode_plan(self, starting_state, path_to_follow):
        self.current_desired_state_index = 0
        self.actions_done_for_current_waypoint = 0
        plan = plan_from_path(path_to_follow, mean_per_stepsize=self.mean_per_stepsize,
                              std_per_stepsize=self.std_per_stepsize,
                              stepsizes_in_waypoint_radii=self.stepsizes_in_waypoint_radii,
                              path_shortcutting=self.path_shortcutting, theta=self.theta,
                              steps_per_waypoint=self.steps_per_waypoint, engine=self.engine)
        self.stds = plan["stds"]
        self.radii = plan["radii"]
        self.distance_function = plan["distance_function"]
        self.path_to_follow = plan["path_to_follow"]
        self.desired_states = plan["desired_states"]
        self.distances_left = plan["distances_left"]
        if self.num_episodes_finished % self.num_episodes_for_aggregation == 0:
            self.train_dynamics_model()
        self.num_episodes_finished += 1
        if len(self.desired_states) >= 2:
            self.engine.set_plan(self.desired_states, self.distances_left, self.radii)

    def close_enough_to_goal(self, current_state):
        if self.distance_function(current_state, self.desired_states[-1]) <= self.theta:
            return True
        return (self.current_desired_state_index == len(self.desired_states) - 1 and
                self.final_steps <= self.actions_done_for_current_waypoint)

    def render(self, env, **kwargs):
        env.render()

    # ------------------------------------------------------------------ model (re)training
    def train_dynamics_model(self):
        """Aggregate replay-buffer transitions with the initial data and fit (NND_MB_agent.py:437-480)."""
        dx, dy = self.dataX.shape[1], self.dataY.shape[1]
        if len(self.replay_buffer) == 0:
            s, a, s2 = np.zeros((0, dx)), np.zeros((0, dy)), np.zeros((0, dx))
        else:
            s, a, _, _, s2 = self.replay_buffer.all_batch()
            s, a, s2 = (np.asarray(v, dtype=np.float64).reshape(len(v), -1) for v in (s, a, s2))
        new_x, new_y, new_z = s, a, s2 - s
        if self.make_aggregated_dataset_noisy and len(s):
            new_x, new_z = self._add_noise(new_x), self._add_noise(new_z)
        with np.errstate(divide="ignore", invalid="ignore"):
            new_x = np.nan_to_num((new_x - self.mean_x) / self.std_x)
            new_y = np.nan_to_num((new_y - self.mean_y) / self.std_y)
            new_z = np.nan_to_num((new_z - self.mean_z) / self.std_z)
        inputs_new = np.concatenate((new_x, new_y), axis=1)
        if self.use_existing_dynamics_model:
            z = np.load(os.path.join(self.load_dir, "models", "finalModel.npz"))
            n = len(self.dyn_model.weights)
            self.dyn_model.set_weights([z["w%d" % i] for i in range(n)], [z["b%d" % i] for i in range(n)])
        else:
            self.dyn_model.train(self.inputs, self.outputs, inputs_new, new_z, self.nEpochs, self.save_dir,
                                 self.fraction_use_new, save_results=self.save_resulting_dynamics_model)
        if self.save_resulting_dynamics_model:
            md = os.path.join(self.save_dir, "models")
            os.makedirs(md, exist_ok=True)
            w, b = self.dyn_model.export()
            blob = {("w%d" % i): wi for i, wi in enumerate(w)}
            blob.update({("b%d" % i): bi for i, bi in enumerate(b)})
            np.savez(os.path.join(md, "model_numTrain%d.npz" %
                                  (1 + self.num_episodes_finished // self.num_episodes_for_aggregation)), **blob)
            np.savez(os.path.join(md, "finalModel.npz"), **blob)

    # ------------------------------------------------------------------ waypoint helpers
    @property
    def current_desired_state(self):
        return self.desired_states[self.current_desired_state_index]

    @property
    def next_desired_state(self):
        return self.desired_states[min(self.current_desired_state_index + 1, len(self.desired_states) - 1)]

    def move_to_next(self, pt, desired_state_index, distance_to_curr, distance_to_next):
        near = np.logical_or(distance_to_curr <= self.theta, distance_to_next <= distance_to_curr)
        return np.logical_and(near, desired_state_index != len(self.desired_states) - 1)
