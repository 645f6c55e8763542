"""Torch restatement of the reference's four learners (SURVEY.md 8(f) row N1).

    DQN        DQN.py:9-443          Flatten -> Dense(50, sigmoid) -> Dense(n_actions), Adam(lr=alpha, clipvalue=1), MSE,
                                     replay deque(memory_size), eps-greedy, target network synced every target_update steps
    DQN_SARSA  DQN_SARSA.py:7-191    on-policy target r + gamma * Q_target(s', a')
    DQN_DUEL   DQN_DUEL.py:13-48     dueling head  Q = V + (A - mean A)
    DQN_BOTH   DQN_BOTH.py:4-8       both (same MRO mix-in as the reference)

Same class names, constructor, methods and log format (``Logs/<name>`` JSON readable by the
reference's analyze.py), so ``main.py -r -t DQN|SARSA|DDQN|BOTH|Baseline`` style loops run against the
CUDA environment: ``sim`` is ``wildfire_control_python_b200.ForestFire`` (or anything with the
reference's ``reset / step / render / W.agents / METADATA`` surface).

What is B200-native here: the environment step is the CUDA path behind the C ABI; the replay memory
lives in device tensors and one ``replay()`` is two batched forward passes of the target network and
one optimiser step (the reference issues 2 x batch_size single-sample ``predict`` calls, DQN.py:164-176).
The learning rule itself is unchanged: the regression target of a sample is the TARGET network's
Q-vector with the taken action's entry replaced (DQN.py:166-176), loss = MSE over all outputs.
Keras is not a dependency; weights are saved as ``.npz`` with Keras' layer names
(``dense_1/kernel:0`` ...), kernels in Keras' [in, out] orientation.
"""
from __future__ import annotations

import ctypes
import json
import os
import math
import random
import time

import numpy as np
import torch
from torch import nn

from .constants import DQN_DEFAULTS


class ReplayMemory:
    """``collections.deque(maxlen=...)`` of transitions (DQN.py:20, :205-206), stored as device tensors.

    ``maxlen=None`` grows without bound, like the plain ``deque()`` collect_memories switches to
    (DQN.py:290).  Sampling is uniform without replacement (``random.sample``, DQN.py:161).
    """

    def __init__(self, obs_shape, device, maxlen=None, with_aprime=False):
        self.maxlen, self.device, self.with_aprime = maxlen, device, with_aprime
        self.obs_shape = tuple(obs_shape)
        self._cap = 0
        self._n = 0       # number of valid entries
        self._head = 0    # position of the oldest entry once the ring is full
        self._grow(min(maxlen, 4096) if maxlen else 4096)

    def _grow(self, cap):
        def buf(shape, dtype):
            t = torch.zeros((cap,) + shape, dtype=dtype, device=self.device)
            return t
        new = dict(s=buf(self.obs_shape, torch.uint8), sp=buf(self.obs_shape, torch.uint8), a=buf((), torch.int64),
                   ap=buf((), torch.int64), r=buf((), torch.float32), d=buf((), torch.bool))
        if self._cap:
            for k, t in new.items():
                t[: self._cap] = getattr(self, "_" + k)
        for k, t in new.items():
            setattr(self, "_" + k, t)
        self._cap = cap

    def __len__(self):
        return self._n

    def _as_obs(self, x):
        t = torch.as_tensor(np.asarray(x) if not torch.is_tensor(x) else x)
        return t.reshape(self.obs_shape).to(device=self.device, dtype=torch.uint8)

    def append(self, state, action, reward, sprime, done, aprime=0):
        if self.maxlen is not None and self._n == self.maxlen:
            i = self._head  # full: the oldest entry is dropped, like deque(maxlen)
            self._head = (self._head + 1) % self.maxlen
        else:
            if self._n == self._cap:
                self._grow(min(2 * self._cap, self.maxlen) if self.maxlen else 2 * self._cap)
            i = self._n
            self._n += 1
        self._s[i] = self._as_obs(state)
        self._sp[i] = self._as_obs(sprime)
        self._a[i], self._ap[i], self._r[i], self._d[i] = int(action), int(aprime), float(reward), bool(done)

    def append_bulk(self, states, actions, rewards, sprimes, dones, aprimes=None):
        """Append M transitions held in device tensors (unbounded memories only)."""
        assert self.maxlen is None
        m = int(actions.shape[0])
        while self._n + m > self._cap:
            self._grow(2 * self._cap)
        sl = slice(self._n, self._n + m)
        self._s[sl] = states.reshape((m,) + self.obs_shape).to(self.device, torch.uint8)
        self._sp[sl] = sprimes.reshape((m,) + self.obs_shape).to(self.device, torch.uint8)
        self._a[sl] = actions.to(self.device, torch.int64)
        self._ap[sl] = 0 if aprimes is None else aprimes.to(self.device, torch.int64)
        self._r[sl] = rewards.to(self.device, torch.float32)
        self._d[sl] = dones.to(self.device, torch.bool)
        self._n += m

    def sample(self, batch_size):
        idx = torch.as_tensor(random.sample(range(self._n), batch_size), device=self.device)
        return (self._s[idx], self._a[idx], self._r[idx], self._sp[idx], self._ap[idx], self._d[idx])


class _QNet(nn.Module):
    """DQN.make_network (DQN.py:209-233): Flatten -> Dense(50, sigmoid) -> Dense(n_actions, linear)."""

    def __init__(self, n_in, n_actions):
        super().__init__()
        self.dense_1 = nn.Linear(n_in, 50)
        self.dense_2 = nn.Linear(50, n_actions)
        _keras_init(self)

    def forward(self, x):
        return self.dense_2(torch.sigmoid(self.dense_1(x.flatten(1))))


class _DuelNet(nn.Module):
    """DQN_DUEL.make_network (DQN_DUEL.py:18-48): advantage and value streams, q = v + (a - mean(a))."""

    def __init__(self, n_in, n_actions):
        super().__init__()
        self.dense_1 = nn.Linear(n_in, 50)       # advantage stream
        self.dense_2 = nn.Linear(50, n_actions)
        self.dense_3 = nn.Linear(n_in, 50)       # value stream
        self.dense_4 = nn.Linear(50, 1)
        _keras_init(self)

    def forward(self, x):
        x = x.flatten(1)
        adv = self.dense_2(torch.sigmoid(self.dense_1(x)))
        val = self.dense_4(torch.sigmoid(self.dense_3(x)))
        return val + (adv - adv.mean(dim=1, keepdim=True))


class KerasAdam(torch.optim.Optimizer):
    """``keras.optimizers.Adam(lr, clipvalue)`` of Keras 2 (the reference's ``Adam(lr=self.alpha, clipvalue=1)``,
    DQN.py:227-230), update for update: every gradient element is clipped to [-clipvalue, clipvalue], then
    ``lr_t = lr * sqrt(1 - beta_2^t) / (1 - beta_1^t)``, ``p -= lr_t * m / (sqrt(v) + epsilon)`` with
    ``epsilon = K.epsilon() = 1e-7`` added to the UNCORRECTED second moment (``torch.optim.Adam`` adds its epsilon after
    the bias correction, i.e. an effective epsilon sqrt(1 - beta_2^t) times smaller).  Pinned by tests/golden/agents/n1_replay.npz."""

    def __init__(self, params, lr=0.001, beta_1=0.9, beta_2=0.999, epsilon=1e-7, clipvalue=None):
        super().__init__(params, dict(lr=lr, beta_1=beta_1, beta_2=beta_2, epsilon=epsilon, clipvalue=clipvalue))

    @torch.no_grad()
    def step(self):
        for group in self.param_groups:
            b1, b2 = group["beta_1"], group["beta_2"]
            for p in group["params"]:
                if p.grad is None:
                    continue
                st = self.state[p]
                if not st:
                    st["t"], st["m"], st["v"] = 0, torch.zeros_like(p), torch.zeros_like(p)
                g = p.grad if group["clipvalue"] is None else p.grad.clamp(-group["clipvalue"], group["clipvalue"])
                st["t"] += 1
                st["m"].mul_(b1).add_(g, alpha=1.0 - b1)
                st["v"].mul_(b2).addcmul_(g, g, value=1.0 - b2)
                lr_t = group["lr"] * math.sqrt(1.0 - b2 ** st["t"]) / (1.0 - b1 ** st["t"])
                p.addcdiv_(st["m"], st["v"].sqrt().add_(group["epsilon"]), value=-lr_t)


def _keras_init(net):
    """Keras Dense defaults: glorot_uniform kernel, zero bias."""
    for m in net.modules():
        if isinstance(m, nn.Linear):
            nn.init.xavier_uniform_(m.weight)
            nn.init.zeros_(m.bias)


class DQN:
    def __init__(self, sim, name="no_name", verbose=True, device=None):
        # Constants and such (DQN.py:10-17)
        self.sim = sim
        self.name = name
        self.METADATA = dict(DQN_DEFAULTS)
        self.METADATA.update(sim.METADATA)
        self.action_size = self.sim.n_actions
        self.DEBUG = getattr(sim, "DEBUG", 1)
        self.verbose = verbose
        if device is None:
            device = getattr(getattr(sim, "_batch", None), "device", None) or ("cuda" if torch.cuda.is_available() else "cpu")
        self.device = torch.device(device)
        self.obs_shape = (self.sim.W.WIDTH, self.sim.W.HEIGHT, self.sim.W.DEPTH)

        # DQN memory (DQN.py:20)
        self.memory = self._new_memory(self.METADATA["memory_size"])

        # Information to save to file (DQN.py:23-32)
        self.logs = {
            "best_reward": -10000,
            "total_rewards": list(),
            "agent_pos": list(),
            "agent_deaths": list(),
            "maps": list(),
            "init_memories": 0,
            "total_time": 0,
            "n_episodes": 0,
        }

        # DQN parameters (DQN.py:35-41)
        self.max_eps = self.METADATA["max_eps"]
        self.min_eps = self.METADATA["min_eps"]
        self.eps_decay_rate = self.METADATA["eps_decay_rate"]
        self.eps = self.max_eps
        self.gamma = self.METADATA["gamma"]
        self.alpha = self.METADATA["alpha"]
        self.target_update_freq = self.METADATA["target_update"]

        # Network and target network (DQN.py:44-46)
        self.model = self.make_network()
        self.target = self.make_network()
        self.target.load_state_dict(self.model.state_dict())
        # Adam(lr=alpha, clipvalue=1), Keras' update rule; loss = mse (DQN.py:227-230)
        self.optimizer = KerasAdam(self.model.parameters(), lr=self.alpha, clipvalue=1.0)

        if self.verbose:
            width, height = self.METADATA["width"], self.METADATA["height"]
            print("\n\t[Parameters]")
            print("[decay]", self.METADATA["eps_decay_rate"])
            print("[alpha]", self.METADATA["alpha"])
            print("[gamma]", self.METADATA["gamma"])
            print("[batch]", self.METADATA["batch_size"])
            print("[size]", f"{width}x{height}")
            print("[wind speed]", self.METADATA["wind"][0] if self.METADATA["wind"] != "random" else "random")
            print("[target upd]", self.METADATA["target_update"], "\n")

    # ------------------------------------------------------------------ learning
    _SARSA = False

    def _new_memory(self, maxlen):
        return ReplayMemory(self.obs_shape, self.device, maxlen=maxlen, with_aprime=self._SARSA)

    def _as_batch(self, state):
        """np.reshape(state, [1] + shape) of the reference; a device float tensor here."""
        t = state if torch.is_tensor(state) else torch.as_tensor(np.asarray(state))
        return t.reshape((1,) + self.obs_shape).to(device=self.device, dtype=torch.float32)

    def learn(self, n_episodes=1000):
        """The training loop of DQN.learn (DQN.py:65-153) and DQN_SARSA.learn (DQN_SARSA.py:12-100): one episode
        after another, one ``replay`` per step once the memory holds more than a batch, target network
        refreshed every ``target_update`` steps, epsilon decayed per episode, logs written at the end.
        The on-policy variant picks the next action BEFORE storing the transition (it is part of it)."""
        t_run = time.time()
        self.logs["n_episodes"] = n_episodes
        until_sync = self.target_update_freq
        batch = self.METADATA["batch_size"]
        for episode in range(n_episodes):
            t_episode = time.time()
            state = self._as_batch(self.sim.reset())
            if self.DEBUG > 0 and not self._SARSA:  # only DQN.learn records the start cell (DQN.py:89-91)
                me = self.sim.W.agents[0]
                self.logs["agent_pos"].append((me.x, me.y))
            action = self.choose_action(state) if self._SARSA else None
            episode_return, done = 0, False
            while not done:
                if not self._SARSA:
                    action = self.choose_action(state)
                observed, reward, done, _ = self.sim.step(action)
                observed = self._as_batch(observed)
                if self._SARSA:
                    upcoming = self.choose_action(observed)
                    self.remember(state, action, reward, observed, upcoming, done)
                else:
                    upcoming = None
                    self.remember(state, action, reward, observed, done)
                if len(self.memory) > batch:
                    self.replay()
                until_sync -= 1
                if until_sync == 0:
                    until_sync = self.target_update_freq
                    self.target.load_state_dict(self.model.state_dict())
                state, action = observed, upcoming
                episode_return += reward
            self._end_of_episode(episode, episode_return, t_episode)
        self.logs["total_time"] = round(time.time() - t_run, 3)
        self.write_data()

    def _end_of_episode(self, episode, total_reward, t0):  # DQN.py:120-148
        dead = len(self.sim.W.agents) == 0
        if self.DEBUG > 0:
            self.logs["agent_deaths"].append(dead)
        if total_reward >= 0.9 * self.logs["best_reward"] or total_reward > 300:
            map_string = self._render_string()
            if total_reward > self.logs["best_reward"]:
                self.logs["best_reward"] = total_reward
            if self.DEBUG > 0:
                self.logs["maps"].append([episode, map_string])
        if self.verbose:
            print(f"[Episode {episode + 1}]\tTime: {round(time.time() - t0, 3)}")
            print(f"\t\tEpsilon: {round(self.eps, 3)}")
            print(f"\t\tAgent dead: {dead}")
            print(f"\t\tReward: {round(total_reward, 0)}\n")
        self.decay_epsilon(episode)
        self.logs["total_rewards"].append(total_reward)

    def _render_string(self):
        try:
            return self.sim.render(print_map=self.verbose)
        except TypeError:
            return self.sim.render()

    def _bootstrap(self, q_next, aprime):
        """Value of S' used in the target: max_a Q_target(S', a) (DQN.py:174-175)."""
        return q_next.max(dim=1).values

    def replay_targets(self, batch):
        """The regression targets of one replay batch (DQN.py:164-180): the target network's Q-vector
        of S with the taken action's entry replaced by r (terminal) or r + gamma * bootstrap(S')."""
        s, a, r, sp, ap, d = batch
        with torch.no_grad():
            pred = self.target(s.float())
            boot = self._bootstrap(self.target(sp.float()), ap)
            upd = torch.where(d, r, r + self.gamma * boot)
            pred[torch.arange(len(a), device=pred.device), a] = upd
        return pred

    def replay(self):  # DQN.py:156-185
        return self.fit_batch(self.memory.sample(self.METADATA["batch_size"]))

    def fit_batch(self, batch):
        """``self.model.fit(states, predictions, epochs=1)`` on one batch of transitions (DQN.py:181-185): with the
        reference's batch_size = 32 = Keras' default mini-batch that is exactly one clipped-Adam update on the MSE."""
        targets = self.replay_targets(batch)
        loss = nn.functional.mse_loss(self.model(batch[0].float()), targets)
        self.optimizer.zero_grad(set_to_none=True)
        loss.backward()
        self.optimizer.step()  # clips every gradient element to [-1, 1] first (clipvalue=1)
        return float(loss.detach())

    def choose_action(self, state, eps=None):  # DQN.py:188-196
        eps_threshold = self.eps if eps is None else eps
        if random.uniform(0, 1) > eps_threshold:
            with torch.no_grad():
                return int(self.model(self._as_batch(state)).argmax(dim=1)[0])
        return int(np.random.choice(self.METADATA["n_actions"]))

    def decay_epsilon(self, episode_num=None):  # DQN.py:199-202
        self.eps = self.min_eps + (self.max_eps - self.min_eps) * np.exp(-self.eps_decay_rate * episode_num)

    def remember(self, state, action, reward, sprime, done):  # DQN.py:205-206
        self.memory.append(state, action, reward, sprime, done)

    def make_network(self):  # DQN.py:209-233
        return _QNet(int(np.prod(self.obs_shape)), self.action_size).to(self.device)

    # ------------------------------------------------------------------ helpers
    def play_optimal(self, eps=0, delay=0.1):  # DQN.py:240-253
        done = False
        total_reward = 0
        state = self.sim.reset()
        while not done:
            self.sim.render()
            self.show_info(self._as_batch(state))
            action = self.choose_action(state, eps=eps)
            state, reward, done, _ = self.sim.step(action)
            total_reward += reward
            time.sleep(delay)
        self.sim.render()
        print(f"Total reward: {total_reward}")
        return total_reward

    def show_info(self, state):  # DQN.py:256-276
        print(f"Wind Speed: {self.sim.W.wind_speed}")
        print(f"Wind direction: {self.sim.W.wind_vector}")
        with torch.no_grad():
            qvals = self.model(self._as_batch(state))[0].cpu().numpy()
        key_map = {0: "N", 1: "S", 2: "E", 3: "W", 4: "D", 5: " "}
        print("| ", end="")
        for idx, val in enumerate(qvals):
            val = round(float(val), 2)
            extra_space = " " if val > 0 else ""
            print(f"{key_map[idx]} : {extra_space}{val:.2f} | ", end="")
            if idx == 1:
                print("\n| ", end="")
        print(f"\nBest Action: {key_map[int(np.argmax(qvals))]}\n")

    def collect_memories(self, num_of_episodes=100, perform_baseline=False):
        """Demonstration data (DQN.py:286-348, DQN_SARSA.py:148-191): the heuristic walk round the fire drives the
        env; an episode's transitions enter the (now unbounded, DQN.py:290) memory only if it pays the
        containment bonus, and it is cut there; stop after ``num_of_episodes`` such episodes.
        ``perform_baseline`` (main.py:60-61): store nothing, play ``num_of_episodes`` whole episodes of the
        heuristic policy and log their returns and deaths."""
        if not num_of_episodes:
            return
        self.memory = self._new_memory(None)
        bonus = self.METADATA["contained_bonus"]
        kept, played = 0, 0
        while True:
            episode, episode_return, done = [], 0, False
            state = self._as_batch(self.sim.reset())
            action = self.choose_randomwalk_action() if self._SARSA else None
            while not done:
                if not self._SARSA:
                    action = self.choose_randomwalk_action()
                observed, reward, done, _ = self.sim.step(action)
                observed = self._as_batch(observed)
                if self._SARSA:
                    upcoming = self.choose_randomwalk_action()
                    episode.append((state, action, reward, observed, upcoming, done))
                else:
                    upcoming = None
                    episode.append((state, action, reward, observed, done))
                state, action = observed, upcoming
                episode_return += reward
                if not perform_baseline and reward == bonus:
                    kept += 1
                    for transition in episode:
                        self.remember(*transition)
                    if kept == num_of_episodes:
                        self.logs["init_memories"] = len(self.memory)
                        return
                    break
            if perform_baseline:
                self.logs["total_rewards"].append(episode_return)
                self.logs["agent_deaths"].append(len(self.sim.W.agents) == 0)
                if self.verbose and played % 100 == 0:
                    print(f"Episode {played}/{num_of_episodes}")
                played += 1
                if played == num_of_episodes:
                    self.logs["n_episodes"] = num_of_episodes
                    break
        self.write_data()

    def collect_memories_batched(self, num_of_episodes=100, n_envs=1024, k_steps=256, seed=0):
        """``collect_memories`` (DQN.py:286-348, DQN_SARSA.py:148-191) over ``n_envs`` environments at once:
        the heuristic walk policy runs ON THE DEVICE (``wf_rollout_policy``), whole rollouts of ``k_steps`` steps
        per launch, and the transitions of the episodes that contain the fire (from their reset up to and
        including the step that pays the containment bonus) are gathered into the replay memory.
        Only episodes that start in the first half of a rollout are considered, so that slow containments
        are not under-represented; an episode still undecided at the end of its rollout is dropped.
        Returns the number of environment steps simulated."""
        from .batched import BatchedForestFire
        from .constants import DQN_DEFAULTS as _D
        if not num_of_episodes:
            return 0
        keys = {k: v for k, v in self.METADATA.items() if k not in _D and k not in ("debug", "a_speed_iter", "seed", "auto_reset")}
        env = BatchedForestFire(n_envs, device=self.device if self.device.type == "cuda" else None, auto_reset=True, seed=seed, **keys)
        bonus = self.METADATA["contained_bonus"]
        self.memory = self._new_memory(None)
        success, simulated = 0, 0
        try:
            while success < num_of_episodes:
                obs0 = env.reset().clone()
                obs, rew, done, acts = env.rollout(k_steps, policy="walk", return_actions=True)
                simulated += k_steps * n_envs
                rew_c, done_c = rew.cpu().numpy(), done.cpu().numpy()
                t_idx, e_idx = [], []
                for i in range(n_envs):
                    bounds = list(np.nonzero(done_c[:, i])[0]) + [k_steps - 1]
                    start = 0
                    for end in bounds:
                        if start >= k_steps // 2 or start > end:
                            break
                        hit = np.nonzero(rew_c[start:end + 1, i] == bonus)[0]
                        if len(hit):
                            t_idx.append(np.arange(start, start + hit[0] + 1))
                            e_idx.append(np.full(hit[0] + 1, i))
                            success += 1
                            if success == num_of_episodes:
                                break
                        start = end + 1
                    if success == num_of_episodes:
                        break
                if t_idx:
                    t = torch.as_tensor(np.concatenate(t_idx), device=obs.device)
                    e = torch.as_tensor(np.concatenate(e_idx), device=obs.device)
                    prev = torch.where((t > 0)[:, None, None, None], obs[(t - 1).clamp(min=0), e], obs0[e])
                    nxt = acts[(t + 1).clamp(max=k_steps - 1), e]
                    self.memory.append_bulk(prev, acts[t, e], rew[t, e], obs[t, e], done[t, e], nxt if self._SARSA else None)
        finally:
            env.close()
        self.logs["init_memories"] = len(self.memory)
        return simulated

    @staticmethod
    def _clockwise_options(ax, ay, mid_x, mid_y):
        """The two moves that keep the agent circling the fire origin clockwise (DQN.py:369-376); actions are
        0 N, 1 S, 2 E, 3 W.  The four half-open quadrants tile the map except the origin itself."""
        if ax >= mid_x and ay > mid_y:
            return (1, 3)
        if ax > mid_x and ay <= mid_y:
            return (1, 2)
        if ax <= mid_x and ay < mid_y:
            return (0, 2)
        if ax < mid_x and ay >= mid_y:
            return (0, 3)
        raise UnboundLocalError("the agent stands on the fire origin: the reference has no move for that cell")

    def choose_randomwalk_action(self, avoid_fire=True):
        """DQN.choose_randomwalk_action (DQN.py:353-389): a random one of the two clockwise moves, redrawn (at most
        11 times) while it would step onto a burning cell.  0 when the agent is gone (SARSA asks anyway)."""
        live = self.sim.W.agents
        if not live:
            return 0
        me = live[0]
        options = self._clockwise_options(me.x, me.y, int(self.sim.W.WIDTH / 2), int(self.sim.W.HEIGHT / 2))
        for attempt in range(12):
            action = options[int(np.random.choice(2))]
            if not avoid_fire or not me.fire_in_direction(action):
                break
        return action

    # ------------------------------------------------------------------ persistence
    out_dir = "."  # Logs/ and Models/ are created below this directory (the reference uses the cwd)

    def write_data(self):  # DQN.py:392-424
        self.logs["metadata"] = self.METADATA
        n_episodes = self.logs["n_episodes"]
        n_episodes = n_episodes / 1000 if n_episodes >= 1000 else 0
        memories = self.logs["init_memories"]
        name = self.sim.get_name(self.sim.W.WIDTH, int(n_episodes), memories, self.name)
        logs_dir, models_dir = os.path.join(self.out_dir, "Logs"), os.path.join(self.out_dir, "Models")
        counter = 0
        while os.path.isfile(os.path.join(logs_dir, name)) or os.path.isfile(os.path.join(models_dir, name + ".npz")):
            if counter > 0:
                name = name[: -len(str(counter))]
            name = name + str(counter)
            counter += 1
        os.makedirs(logs_dir, exist_ok=True)
        os.makedirs(models_dir, exist_ok=True)
        self.save_model(name)
        with open(os.path.join(logs_dir, name), "w") as file:
            json.dump(self.logs, file, default=_jsonable)
        return name

    def get_weights(self):
        """Keras-style weight dict: ``dense_k/kernel:0`` [in, out] and ``dense_k/bias:0``."""
        out = {}
        for lname, m in self.model.named_children():
            out[f"{lname}/kernel:0"] = m.weight.detach().t().contiguous().cpu().numpy()
            out[f"{lname}/bias:0"] = m.bias.detach().cpu().numpy()
        return out

    def set_weights(self, weights):
        with torch.no_grad():
            for lname, m in self.model.named_children():
                m.weight.copy_(torch.as_tensor(np.asarray(weights[f"{lname}/kernel:0"])).t())
                m.bias.copy_(torch.as_tensor(np.asarray(weights[f"{lname}/bias:0"])))
        self.target.load_state_dict(self.model.state_dict())

    def load_keras_weights(self, path):
        """Load a network trained by the REFERENCE: a Keras ``save_weights`` HDF5 file from its ``Models/``
        tree (DQN.py:441-443), read without h5py/Keras by ``keras_h5.read_keras_weights``."""
        from .keras_h5 import canonical_dense_names, read_keras_weights
        self.set_weights(canonical_dense_names(read_keras_weights(path)))

    def evaluate_batched(self, n_envs=4096, episodes_per_env=1, eps=None, seed=0, max_steps=100000, in_kernel=None):
        """Roll the current policy out on ``n_envs`` CUDA environments at once (eps-greedy, DQN.py:188-196) and
        return (total reward, agent died) of the first ``episodes_per_env`` episodes of every env -- the
        quantity ``logs['total_rewards']`` / ``logs['agent_deaths']`` hold per training episode.

        ``in_kernel`` (default: whenever the grid fits the warp kernel family, <= 32x32): the Q-network is
        evaluated INSIDE the step kernel (``wf_rollout_policy(WF_POLICY_MLP)``), 64 steps per launch;
        otherwise torch evaluates it between two ``wf_step`` calls.  On grids larger than 32x32 ``in_kernel=True`` is
        the fast path (the tile kernel's policy pass); the default stays the torch path there, whose exploration draws
        come from another random stream, so its results are unchanged."""
        from .batched import BatchedForestFire
        from .constants import DQN_DEFAULTS as _D
        eps = self.min_eps if eps is None else eps
        keys = {k: v for k, v in self.METADATA.items() if k not in _D and k not in ("debug", "a_speed_iter", "seed", "auto_reset")}
        env = BatchedForestFire(n_envs, device=self.device, auto_reset=True, seed=seed, **keys)
        if in_kernel is None:
            in_kernel = env.kernel_family == "warp"
        if in_kernel:
            try:
                return self._evaluate_in_kernel(env, n_envs, episodes_per_env, eps, max_steps)
            finally:
                env.close()
        dev = self.device
        gen = torch.Generator(device=dev).manual_seed(seed)
        returns = torch.zeros((n_envs, episodes_per_env), dtype=torch.float64, device=dev)
        died = torch.zeros((n_envs, episodes_per_env), dtype=torch.bool, device=dev)
        acc = torch.zeros(n_envs, dtype=torch.float64, device=dev)
        n_done = torch.zeros(n_envs, dtype=torch.int64, device=dev)
        rows = torch.arange(n_envs, device=dev)
        death_penalty = float(self.METADATA["death_penalty"])
        try:
            obs = env.reset()
            for step in range(max_steps):
                with torch.no_grad():
                    greedy = self.model(obs.float()).argmax(dim=1).to(torch.int32)
                explore = torch.rand(n_envs, device=dev, generator=gen) < eps
                rnd = torch.randint(0, self.action_size, (n_envs,), device=dev, dtype=torch.int32, generator=gen)
                obs, rew, done, _ = env.step(torch.where(explore, rnd, greedy))
                acc += rew
                live = done & (n_done < episodes_per_env)
                slot = n_done.clamp(max=episodes_per_env - 1)
                returns[rows[live], slot[live]] = acc[live]
                died[rows[live], slot[live]] = rew[live] == death_penalty
                acc = torch.where(done, torch.zeros_like(acc), acc)
                n_done += done.to(torch.int64)
                if step % 16 == 15 and bool((n_done >= episodes_per_env).all()):
                    break
            else:
                raise RuntimeError("evaluate_batched: some episodes did not finish")
        finally:
            env.close()
        return returns.flatten().cpu().numpy(), died.flatten().cpu().numpy()

    def _evaluate_in_kernel(self, env, n_envs, episodes_per_env, eps, max_steps, chunk=64):
        w = self.get_weights()  # dense_1 / dense_2 are the advantage stream of a dueling head: argmax Q = argmax A
        env.set_policy_mlp(w["dense_1/kernel:0"], w["dense_1/bias:0"], w["dense_2/kernel:0"], w["dense_2/bias:0"], eps=eps)
        env.reset()
        death_penalty = float(self.METADATA["death_penalty"])
        returns = np.zeros((n_envs, episodes_per_env))
        died = np.zeros((n_envs, episodes_per_env), dtype=bool)
        n_done = np.zeros(n_envs, dtype=np.int64)
        carry = np.zeros(n_envs)  # reward of the running episode before this chunk
        for _ in range(0, max_steps, chunk):
            _, rew, done = env.rollout(chunk, policy="mlp", obs=False)
            rew, done = rew.cpu().numpy(), done.cpu().numpy()
            e_idx, k_idx, ret, carry = _episode_ends(carry, rew, done)
            same = np.r_[False, e_idx[1:] == e_idx[:-1]]
            first = np.r_[True, ~same[1:]] if len(e_idx) else np.zeros(0, bool)
            rank = np.arange(len(e_idx)) - np.maximum.accumulate(np.where(first, np.arange(len(e_idx)), 0))
            slot = n_done[e_idx] + rank
            keep = slot < episodes_per_env
            returns[e_idx[keep], slot[keep]] = ret[keep]
            died[e_idx[keep], slot[keep]] = rew[k_idx[keep], e_idx[keep]] == death_penalty
            n_done += np.bincount(e_idx, minlength=n_envs)
            if (n_done >= episodes_per_env).all():
                return returns.flatten(), died.flatten()
        raise RuntimeError("evaluate_batched: some episodes did not finish")

    # ------------------------------------------------------------------ batched learning on the device
    def _flat_shape(self, batch):
        from . import _lib
        W, H = self.obs_shape[0], self.obs_shape[1]
        return _lib.WfMlpShape(width=W, height=H, hidden=self.model.dense_1.out_features, n_actions=self.action_size,
                               dueling=int(hasattr(self.model, "dense_3")), batch=int(batch))

    def fit_batches_fused(self, frames, s_row, sp_row, a, ap, r, d, n_replays, phase=None):
        """``n_replays`` consecutive ``fit_batch`` updates in ONE kernel launch (include/wildfire.h), the same rule (targets
        from the target network, MSE, clipped Keras Adam) on packed observations: ``wf_replay_fit`` on grids up to 32x32,
        ``wf_replay_fit_large`` (the whole GPU, first layer cut into column chunks) on larger grids.

        ``frames``: ``[n_frames, words]`` int32 CUDA tensor of ``WF_OBS_BITS`` rows (``pack_obs`` / ``obs_dtype="bits"``);
        ``s_row`` / ``sp_row``: int64 row numbers of S and S'; ``a`` / ``ap``: actions and next actions (``ap`` is used by
        the on-policy learners only); ``r``: rewards; ``d``: done flags -- each of length ``n_replays * batch``, replay i
        taking entries ``i * batch ...``.  A row outside ``frames`` is an all-zero observation, an action outside
        ``[0, n_actions)`` replaces no target entry, an out-of-range next action bootstraps nothing.
        The target network is refreshed every ``target_update`` replays as in ``learn``: ``phase`` (default: carried over
        from the previous call, starting at ``target_update``) is the number of replays left until the next refresh.
        ``model``, ``target`` and the optimiser's ``t``, ``m``, ``v`` are updated in place; returns the ``[n_replays]``
        float32 losses (a device tensor: nothing is synchronised)."""
        from torch.nn.utils import parameters_to_vector
        from . import _lib
        from .batched import _ptr
        if self.device.type != "cuda":
            raise _lib.WildfireError("fit_batches_fused needs a CUDA device (no CPU fallback)")
        n_replays = int(n_replays)
        if n_replays < 1 or len(s_row) % n_replays:
            raise ValueError("the number of transitions must be a positive multiple of n_replays")
        batch = len(s_row) // n_replays
        dev = self.device
        frames = frames.to(dev).contiguous()
        if frames.dtype != torch.int32 or frames.dim() != 2:
            raise ValueError("frames must be an int32 [n_frames, words] tensor")
        cols = [torch.as_tensor(x, device=dev).to(dt).contiguous()
                for x, dt in ((s_row, torch.int64), (sp_row, torch.int64), (a, torch.int32), (ap, torch.int32),
                              (r, torch.float32), (d, torch.uint8))]
        if any(c.shape != (n_replays * batch,) for c in cols):
            raise ValueError("s_row, sp_row, a, ap, r and d must be one-dimensional and of the same length")
        s_row, sp_row, a, ap, r, d = cols
        params = list(self.model.parameters())
        states = [self.optimizer.state[p] for p in params]
        t0 = states[0]["t"] if states[0] else 0
        with torch.no_grad():
            flat = parameters_to_vector(params).contiguous()
            tgt = parameters_to_vector(self.target.parameters()).contiguous()
            m = parameters_to_vector([st["m"] for st in states]) if t0 else torch.zeros_like(flat)
            v = parameters_to_vector([st["v"] for st in states]) if t0 else torch.zeros_like(flat)
        group = self.optimizer.param_groups[0]
        te = int(self.target_update_freq)
        phase = int(getattr(self, "_until_sync", te) if phase is None else phase)
        hp = _lib.WfFitParams(gamma=float(self.gamma), lr=group["lr"], beta_1=group["beta_1"], beta_2=group["beta_2"],
                              epsilon=group["epsilon"], clipvalue=math.inf if group["clipvalue"] is None else group["clipvalue"],
                              adam_t=t0, target_every=te, phase=phase)
        loss = torch.empty(n_replays, dtype=torch.float32, device=dev)
        W, H = self.obs_shape[0], self.obs_shape[1]
        fit = _lib.lib().wf_replay_fit if W <= 32 and H <= 32 else _lib.lib().wf_replay_fit_large
        with torch.cuda.device(dev):
            _lib.check(fit(
                ctypes.byref(self._flat_shape(batch)), ctypes.byref(hp), n_replays, _ptr(flat), _ptr(tgt), _ptr(m), _ptr(v),
                _ptr(frames), frames.shape[0], _ptr(s_row), _ptr(sp_row), _ptr(a), _ptr(ap) if self._SARSA else None,
                _ptr(r), _ptr(d), _ptr(loss), ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
        with torch.no_grad():
            off = 0
            for p, tp, st in zip(params, self.target.parameters(), states):
                n = p.numel()
                p.copy_(flat[off:off + n].view_as(p))
                tp.copy_(tgt[off:off + n].view_as(p))
                st["m"] = m[off:off + n].view_as(p).clone()
                st["v"] = v[off:off + n].view_as(p).clone()
                st["t"] = t0 + n_replays
                off += n
        self._until_sync = (phase - n_replays - 1) % te + 1
        return loss

    def learn_batched(self, n_episodes, n_envs=1024, k_steps=16, replays_per_launch=None, batch_size=None, seed=0,
                      replay_seed=None):
        """``learn`` over ``n_envs`` CUDA environments at once: the envs act with the eps-greedy Q-network evaluated inside
        the step kernel (``rollout(policy="mlp")``, ``k_steps`` steps per launch), each rollout writes its packed
        observations straight into a device replay ring, and after every launch ``replays_per_launch`` (default
        ``k_steps``) replays of ``batch_size`` (default METADATA's) transitions run as one ``fit_batches_fused`` launch.
        The in-kernel policy is refreshed on the device before every launch, with eps = min + (max - min) *
        exp(-rate * episodes completed so far) (``decay_epsilon``).

        Replay memory: the ring (``_PackedReplayRing``) holds at least the last ``memory_size`` transitions of every env
        together (whole launches, at least two), plus every transition already in ``self.memory`` (demonstrations from ``collect_memories(_batched)``, kept for
        the whole run like the reference's unbounded post-demonstration deque).  Each replay draws its batch uniformly
        without replacement from both, on the device, from a generator seeded with ``replay_seed`` (default: ``seed``, the
        envs' Philox key); replays start once more
        than a batch of transitions exists.  The target network is refreshed every ``target_update`` replays.

        Runs until ``n_episodes`` episodes have ended (over all envs, in order of their last step, then env) and logs those
        in the reference's format (``total_rewards``, ``agent_deaths``, ``n_episodes``, ``init_memories``,
        ``total_time``; ``write_data``).  Per-episode ``maps`` and ``agent_pos`` are not recorded: the envs run on the
        device and are not rendered.  One small device-to-host read per launch (rewards and done flags).
        ``eps_per_launch`` / ``episodes_before_launch`` record the schedule.  Any grid: ``fit_batches_fused`` runs the
        replays in ``wf_replay_fit`` up to 32x32 and in ``wf_replay_fit_large`` on larger grids.  Returns the number of
        environment steps simulated."""
        from .batched import BatchedForestFire
        from .constants import DQN_DEFAULTS as _D
        t_run = time.time()
        N, K = int(n_envs), int(k_steps)
        R = K if replays_per_launch is None else int(replays_per_launch)
        B = int(self.METADATA["batch_size"] if batch_size is None else batch_size)
        keys = {k: v for k, v in self.METADATA.items() if k not in _D and k not in ("debug", "a_speed_iter", "seed", "auto_reset")}
        env = BatchedForestFire(N, device=self.device, obs_dtype="bits", auto_reset=True, seed=seed, **keys)
        death_penalty = float(self.METADATA["death_penalty"])
        gen = torch.Generator(device=env.device).manual_seed(int(seed if replay_seed is None else replay_seed))
        self._until_sync = self.target_update_freq
        self.logs["n_episodes"] = n_episodes
        self.eps_per_launch, self.episodes_before_launch = [], []
        rewards, deaths = [], []
        carry = np.zeros(N)
        done_eps = 0
        try:
            ring = _PackedReplayRing(env, K, int(self.METADATA["memory_size"]), self.memory, self._SARSA)
            while len(rewards) < n_episodes:
                self.eps = self.min_eps + (self.max_eps - self.min_eps) * np.exp(-self.eps_decay_rate * done_eps)
                self.eps_per_launch.append(float(self.eps))
                self.episodes_before_launch.append(done_eps)
                net = self.model
                env.set_policy_mlp_dev(net.dense_1.weight, net.dense_1.bias, net.dense_2.weight, net.dense_2.bias, eps=self.eps)
                rew, done = ring.launch()
                if R > 0 and ring.n_sampleable > B:
                    self.fit_batches_fused(ring.frames, *ring.gather(ring.sample(R, B, gen)), R)
                rd = torch.stack((rew, done.double())).cpu().numpy()
                e_idx, k_idx, ret, carry = _episode_ends(carry, rd[0], rd[1] != 0)
                order = np.lexsort((e_idx, k_idx))
                for i in order[: n_episodes - len(rewards)]:
                    rewards.append(float(ret[i]))
                    deaths.append(bool(rd[0][k_idx[i], e_idx[i]] == death_penalty))
                done_eps += len(e_idx)
            steps = ring.steps
        finally:
            env.close()
        self.logs["total_rewards"] = rewards
        self.logs["agent_deaths"] = deaths
        self.logs["total_time"] = round(time.time() - t_run, 3)
        self.write_data()
        return steps * N

    def save_model(self, name):  # DQN.py:441-443
        path = os.path.join(self.out_dir, "Models", name)
        np.savez(path, **self.get_weights())
        return path + ".npz"

    def load_model(self, path=None):  # DQN.py:427-438 (interactive when no path is given)
        if path is None:
            all_names = sorted(os.listdir(os.path.join(self.out_dir, "Models")))
            print("\nChoose a model from the list below to load:")
            for idx, n in enumerate(all_names):
                print(f"\t[{idx}] {n}")
            try:
                path = os.path.join(self.out_dir, "Models", all_names[int(input(f"Select one [0-{len(all_names) - 1}]: \n"))])
            except (ValueError, IndexError):
                print("Invalid Selection")
                return
        with np.load(path) as z:
            self.set_weights({k: z[k] for k in z.files})
        if self.verbose:
            print("Model loaded!")


class _PackedReplayRing:
    """The device replay memory of ``DQN.learn_batched`` and ``learn_population``: every rollout of a ``"bits"`` env writes
    its observations, actions, rewards and done flags straight into the next ``K`` slots of a ``[T][N]`` ring; transitions
    are addressed by rows of one ``frames`` table, ``[ring T*N | the frames before the first step N | per group j:
    demonstration s D_j | s' D_j]``.

    The N envs form ``groups`` equal column groups of G = N / groups envs, one per learner: group j's transitions are
    those of envs j*G ... j*G + G - 1, plus its own demonstrations.  ``learn_batched`` is the one-group case.
    Transition (t, n) of global step t and env n: s = the frame of step t - 1 (after an auto-reset already the new
    episode's start; the reset frame for t = 0), a / r / done / s' of step t, a' = the action of step t + 1 (so an
    on-policy transition becomes sampleable one step later).  Held after ``steps`` steps: t in [lo, hi) with
    lo = max(0, steps - T + 1) (s of step lo is the oldest frame the ring holds) and hi = steps (steps - 1 with a').
    T is the smallest multiple of K, and at least 2K, for which T - 1 (T - 2 with a') steps of a group's G envs hold
    ``memory_size`` transitions.  The demonstrations (``ReplayMemory`` entries, uint8; ``demos``: one memory per group, or
    one memory for one group) are packed once and kept."""

    def __init__(self, env, k_steps, memory_size, demos, on_policy, groups=1):
        from .batched import pack_obs
        self.env, self.K, self.N, self.on_policy = env, int(k_steps), env.n_envs, bool(on_policy)
        if not isinstance(demos, (list, tuple)):
            demos = [demos]
        if len(demos) != groups or self.N % groups:
            raise ValueError("need one demonstration memory per group and equal groups of envs")
        self.G = G = self.N // groups
        K, N, dev, words = self.K, self.N, env.device, env.obs_words
        need = -(-int(memory_size) // G) + 1 + int(self.on_policy)
        self.T = T = max(2, -(-need // K)) * K
        self.D = [len(m) for m in demos]
        self.demo_base = [T * N + N + 2 * sum(self.D[:j]) for j in range(groups)]  # first row of group j's demo s
        self.frames = torch.zeros((T * N + N + 2 * sum(self.D), words), dtype=torch.int32, device=dev)
        self.ring = self.frames[: T * N].view(T, N, words)
        self.acts = torch.zeros((T, N), dtype=torch.int32, device=dev)
        self.rews = torch.zeros((T, N), dtype=torch.float64, device=dev)
        self.dones = torch.zeros((T, N), dtype=torch.uint8, device=dev)
        self.demo = []
        for m, D, base in zip(demos, self.D, self.demo_base):
            if D:
                self.frames[base:base + D] = pack_obs(m._s[:D])
                self.frames[base + D:base + 2 * D] = pack_obs(m._sp[:D])
            self.demo.append((m._a[:D].to(torch.int32), m._ap[:D].to(torch.int32), m._r[:D].float(),
                              m._d[:D].to(torch.uint8)) if D else None)
        self.steps = 0
        self.frames[T * N:T * N + N] = env.reset()

    def launch(self):
        """One ``rollout(K, policy="mlp")`` into the next K slots; returns its rewards [K, N] and done flags [K, N]."""
        sl = slice(self.steps % self.T, self.steps % self.T + self.K)
        _, _, _, chosen = self.env.rollout(self.K, policy="mlp", return_actions=True,
                                           out=(self.ring[sl], self.rews[sl], self.dones[sl]))
        self.acts[sl] = chosen
        self.steps += self.K
        return self.rews[sl], self.dones[sl]

    @property
    def window(self):
        """Global steps [lo, hi) whose transitions are held."""
        return max(0, self.steps - self.T + 1), self.steps - int(self.on_policy)

    def sampleable(self, group=0):
        """Transitions group ``group`` can draw from: its envs' held transitions and its demonstrations."""
        lo, hi = self.window
        return max(0, hi - lo) * self.G + self.D[group]

    @property
    def n_sampleable(self):
        return self.sampleable(0)

    def sample(self, n_batches, batch, gen, group=0):
        """``n_batches`` batches, each drawn uniformly without replacement from the group's sampleable transitions:
        [n * batch]."""
        return torch.rand((n_batches, self.sampleable(group)), device=self.frames.device, generator=gen).topk(batch, dim=1).indices.flatten()

    def gather(self, k, group=0):
        """Transitions k of group ``group`` (0 .. sampleable - 1: its ring transitions (t, n) in order of t then n, then
        its demonstrations) as ``fit_batches_fused``'s (s_row, sp_row, a, ap, r, d), rows of the shared ``frames``."""
        T, N, G, D = self.T, self.N, self.G, self.D[group]
        lo, hi = self.window
        nv = max(0, hi - lo) * G
        ring_k = k.clamp(max=max(nv - 1, 0))
        t, n = lo + ring_k // G, ring_k % G + group * G
        slot, prev, nxt = t % T, (t - 1) % T, (t + 1) % T
        s_row = torch.where(t == 0, T * N + n, prev * N + n)
        sp_row = slot * N + n
        a, ap, r, d = self.acts[slot, n], self.acts[nxt, n], self.rews[slot, n].float(), self.dones[slot, n]
        if D:
            base = self.demo_base[group]
            is_demo = k >= nv
            j = (k - nv).clamp(min=0, max=D - 1)
            s_row = torch.where(is_demo, base + j, s_row)
            sp_row = torch.where(is_demo, base + D + j, sp_row)
            a, ap, r, d = (torch.where(is_demo, x[j], y) for x, y in zip(self.demo[group], (a, ap, r, d)))
        return s_row, sp_row, a, ap, r, d


# METADATA keys the learners of one learn_population may set differently: the learning rate, the discount, the target
# refresh interval and the eps schedule.  Everything else (the environment, memory_size, batch_size) must agree.
_POPULATION_FREE_KEYS = ("alpha", "gamma", "target_update", "max_eps", "min_eps", "eps_decay_rate")


def learn_population(agents, n_episodes, envs_per_learner=64, k_steps=16, replays_per_launch=None, batch_size=None, seed=0):
    """``DQN.learn_batched`` for M = len(agents) independent learners (1 to 64) at once on one GPU, with one rollout launch
    and one ``wf_replay_fit_many`` launch per iteration for all of them.

    The agents must be of one class and share the network shape, the environment METADATA, ``memory_size`` and the batch
    size; their initial weights, demonstrations already in ``agent.memory``, ``alpha``, ``gamma``, ``target_update`` and
    eps schedule may differ.  One ``"bits"`` handle of M * ``envs_per_learner`` auto-reset envs with Philox key ``seed``
    runs them all: learner j's envs are the j-th group of ``envs_per_learner`` (a multiple of 8), acting with learner j's
    network and eps (``set_policy_mlp_flat_dev``).  The replay ring (``_PackedReplayRing``) keeps one column group and
    the demonstrations per learner; learner j draws its batches from its own window with its own generator, seeded with
    ``seed + j``.  The stacked [M, P] model, target and Adam moments are the state during the run and are written back
    into each agent (modules, ``KerasAdam`` m, v and t, ``_until_sync``) at the end.

    Learner j logs its first ``n_episodes`` episodes exactly as ``learn_batched`` does (``eps_per_launch`` and
    ``episodes_before_launch`` included) and stops replaying after the launch in which it reaches them; its envs keep
    stepping, ignored, until every learner has finished.  Then each agent calls ``write_data()``.  Agent j's result is
    that of ``agent.learn_batched(n_episodes, envs_per_learner, k_steps, replays_per_launch, batch_size, seed=seed,
    replay_seed=seed + j)`` with METADATA ``env_id_base = j * envs_per_learner``, byte for byte.
    Returns the env-step count of each learner (what ``learn_batched`` returns)."""
    from torch.nn.utils import parameters_to_vector
    from . import _lib
    from .batched import BatchedForestFire, _ptr
    from .constants import DQN_DEFAULTS as _D
    agents = list(agents)
    M = len(agents)
    if not 1 <= M <= _lib.MAX_LEARNERS:
        raise ValueError(f"learn_population takes 1 to {_lib.MAX_LEARNERS} agents, got {M}")
    a0 = agents[0]
    if any(type(a) is not type(a0) for a in agents):
        raise ValueError("learn_population: every agent must be of the same class")
    shared = lambda a: {k: v for k, v in a.METADATA.items() if k not in _POPULATION_FREE_KEYS}
    if any(shared(a) != shared(a0) for a in agents):
        raise ValueError("learn_population: the agents' METADATA (environment, memory_size, batch_size) must agree")
    shapes = lambda a: [tuple(p.shape) for p in a.model.parameters()]
    if any(shapes(a) != shapes(a0) for a in agents):
        raise ValueError("learn_population: every agent must have the same network shape")
    W, H = a0.obs_shape[0], a0.obs_shape[1]
    if W > 32 or H > 32:
        raise ValueError("learn_population runs the in-kernel policy: grids up to 32x32 only")
    G, K = int(envs_per_learner), int(k_steps)
    if G < 8 or G % 8:
        raise ValueError("envs_per_learner must be a positive multiple of 8")
    if any(a.device != a0.device for a in agents):
        raise ValueError("learn_population: every agent must be on the same device")
    if a0.device.type != "cuda":
        raise _lib.WildfireError("learn_population needs a CUDA device (no CPU fallback)")
    t_run = time.time()
    N = M * G
    R = K if replays_per_launch is None else int(replays_per_launch)
    B = int(a0.METADATA["batch_size"] if batch_size is None else batch_size)
    sarsa, dueling = a0._SARSA, hasattr(a0.model, "dense_3")
    hidden = a0.model.dense_1.out_features
    keys = {k: v for k, v in a0.METADATA.items() if k not in _D and k not in ("debug", "a_speed_iter", "seed", "auto_reset")}
    env = BatchedForestFire(N, device=a0.device, obs_dtype="bits", auto_reset=True, seed=seed, **keys)
    dev = env.device
    death_penalty = float(a0.METADATA["death_penalty"])
    gens = [torch.Generator(device=dev).manual_seed(int(seed) + j) for j in range(M)]
    # the stacked state, as DQN.fit_batches_fused flattens it
    with torch.no_grad():
        adam_t = [(a.optimizer.state[next(a.model.parameters())] or {}).get("t", 0) for a in agents]
        P = torch.stack([parameters_to_vector(a.model.parameters()) for a in agents]).contiguous()
        Tg = torch.stack([parameters_to_vector(a.target.parameters()) for a in agents]).contiguous()
        Mm = torch.stack([parameters_to_vector([a.optimizer.state[p]["m"] for p in a.model.parameters()]) if t else
                          torch.zeros(P.shape[1], device=dev) for a, t in zip(agents, adam_t)]).contiguous()
        Vv = torch.stack([parameters_to_vector([a.optimizer.state[p]["v"] for p in a.model.parameters()]) if t else
                          torch.zeros(P.shape[1], device=dev) for a, t in zip(agents, adam_t)]).contiguous()
    until_sync = [int(a.target_update_freq) for a in agents]
    rewards, deaths = [[] for _ in agents], [[] for _ in agents]
    carry = [np.zeros(G) for _ in agents]
    done_eps, steps, finished = [0] * M, [0] * M, [False] * M
    for a in agents:
        a.logs["n_episodes"] = n_episodes
        a.eps_per_launch, a.episodes_before_launch = [], []
    shape = a0._flat_shape(B)
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    try:
        ring = _PackedReplayRing(env, K, int(a0.METADATA["memory_size"]), [a.memory for a in agents], sarsa, groups=M)
        while not all(finished):
            for j, a in enumerate(agents):
                if not finished[j]:
                    a.eps = a.min_eps + (a.max_eps - a.min_eps) * np.exp(-a.eps_decay_rate * done_eps[j])
                    a.eps_per_launch.append(float(a.eps))
                    a.episodes_before_launch.append(done_eps[j])
            env.set_policy_mlp_flat_dev(P, hidden, dueling, [float(a.eps) for a in agents])
            rew, done = ring.launch()
            fit = [j for j in range(M) if not finished[j] and R > 0 and ring.sampleable(j) > B]
            if fit:
                keep, desc = [], (_lib.WfFitLearner * len(fit))()
                for i, j in enumerate(fit):
                    a = agents[j]
                    cols = [x.to(dt).contiguous() for x, dt in zip(ring.gather(ring.sample(R, B, gens[j], j), j),
                                                                   (torch.int64, torch.int64, torch.int32, torch.int32,
                                                                    torch.float32, torch.uint8))]
                    keep.append(cols)
                    grp = a.optimizer.param_groups[0]
                    te = int(a.target_update_freq)
                    hp = _lib.WfFitParams(gamma=float(a.gamma), lr=grp["lr"], beta_1=grp["beta_1"], beta_2=grp["beta_2"],
                                          epsilon=grp["epsilon"],
                                          clipvalue=math.inf if grp["clipvalue"] is None else grp["clipvalue"],
                                          adam_t=adam_t[j], target_every=te, phase=until_sync[j])
                    desc[i] = _lib.WfFitLearner(P[j].data_ptr(), Tg[j].data_ptr(), Mm[j].data_ptr(), Vv[j].data_ptr(),
                                                cols[0].data_ptr(), cols[1].data_ptr(), cols[2].data_ptr(),
                                                cols[3].data_ptr() if sarsa else None, cols[4].data_ptr(),
                                                cols[5].data_ptr(), None, hp)
                with torch.cuda.device(dev):
                    _lib.check(_lib.lib().wf_replay_fit_many(ctypes.byref(shape), len(fit), desc, R, _ptr(ring.frames),
                                                             ring.frames.shape[0], stream))
                for j in fit:
                    adam_t[j] += R
                    te = int(agents[j].target_update_freq)
                    until_sync[j] = (until_sync[j] - R - 1) % te + 1
            rd = torch.stack((rew, done.double())).cpu().numpy()
            for j in range(M):
                if finished[j]:
                    continue
                cols = slice(j * G, (j + 1) * G)
                e_idx, k_idx, ret, carry[j] = _episode_ends(carry[j], rd[0][:, cols], rd[1][:, cols] != 0)
                order = np.lexsort((e_idx, k_idx))
                for i in order[: n_episodes - len(rewards[j])]:
                    rewards[j].append(float(ret[i]))
                    deaths[j].append(bool(rd[0][k_idx[i], j * G + e_idx[i]] == death_penalty))
                done_eps[j] += len(e_idx)
                if len(rewards[j]) >= n_episodes:
                    finished[j], steps[j] = True, ring.steps * G
    finally:
        env.close()
    total_time = round(time.time() - t_run, 3)
    with torch.no_grad():
        for j, a in enumerate(agents):
            params = list(a.model.parameters())
            off = 0
            for p, tp in zip(params, a.target.parameters()):
                n = p.numel()
                p.copy_(P[j, off:off + n].view_as(p))
                tp.copy_(Tg[j, off:off + n].view_as(p))
                if adam_t[j]:
                    st = a.optimizer.state[p]
                    st["m"] = Mm[j, off:off + n].view_as(p).clone()
                    st["v"] = Vv[j, off:off + n].view_as(p).clone()
                    st["t"] = adam_t[j]
                off += n
            a._until_sync = until_sync[j]
            a.logs["total_rewards"] = rewards[j]
            a.logs["agent_deaths"] = deaths[j]
            a.logs["total_time"] = total_time
            a.write_data()
    return steps


def _episode_ends(carry, rew, done):
    """Episodes that end within a [K, N] chunk of rewards and done flags: (env, step, return) of each, sorted by env then
    step, and the new carry (reward of each env's running episode at the end of the chunk; ``carry`` is the one before)."""
    c = carry[None, :] + np.cumsum(rew, axis=0)
    e_idx, k_idx = np.nonzero(done.T)  # episode ends, sorted by env then step
    at_end = c[k_idx, e_idx]
    same = np.r_[False, e_idx[1:] == e_idx[:-1]]
    ret = at_end - np.where(same, np.r_[0.0, at_end[:-1]], 0.0)
    last = np.zeros(len(carry))
    if len(e_idx):
        is_last = np.r_[e_idx[1:] != e_idx[:-1], True]
        last[e_idx[is_last]] = at_end[is_last]
    return e_idx, k_idx, ret, c[-1] - last


def _jsonable(o):
    if isinstance(o, (np.integer,)):
        return int(o)
    if isinstance(o, (np.floating,)):
        return float(o)
    if isinstance(o, np.ndarray):
        return o.tolist()
    if isinstance(o, (np.bool_,)):
        return bool(o)
    raise TypeError(f"not JSON serialisable: {type(o)}")


class DQN_SARSA(DQN):
    _SARSA = True

    def __init__(self, sim, name="no_name", verbose=True, device=None):
        DQN.__init__(self, sim, name, verbose, device)

    def _bootstrap(self, q_next, aprime):
        """On-policy value of S': Q_target(S', A') (DQN_SARSA.py:120-121)."""
        return q_next.gather(1, aprime[:, None])[:, 0]

    def remember(self, state, action, reward, sprime, aprime, done):  # DQN_SARSA.py:134-135
        self.memory.append(state, action, reward, sprime, done, aprime)

    def collect_memories(self, num_of_successes=100):  # DQN_SARSA.py:148-191 (no baseline mode there)
        return DQN.collect_memories(self, num_of_successes, perform_baseline=False)


class DQN_DUEL(DQN):
    def __init__(self, sim, name="no_name", verbose=True, device=None):
        DQN.__init__(self, sim, name, verbose, device)

    def make_network(self):  # DQN_DUEL.py:18-48
        return _DuelNet(int(np.prod(self.obs_shape)), self.action_size).to(self.device)


class DQN_BOTH(DQN_SARSA, DQN_DUEL):  # DQN_BOTH.py:4-8
    def __init__(self, sim, name="no_name", verbose=True, device=None):
        DQN_SARSA.__init__(self, sim, name, verbose, device)
