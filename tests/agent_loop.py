"""The reference's control loop around the hot path, for drop-in tests (BASELINE configs[0]/[2] with a synthetic
environment; VERDICT r1 N2).

Two interchangeable drivers produce the same :class:`Trace`:

  * :func:`run_reference_loop` — the REFERENCE's own `Agent` + `Statistics` (src/agent.py, src/statistics.py,
    converted in a temp dir by tests/ref_convert.py) driven through the schedule of src/main.py:130-162; it needs a
    checkout of the original project and produces tests/golden/agent_loop_golden.npz (make_agent_golden.py);
  * :func:`run_restated_loop` — an independent restatement of that loop written for this repository.
    tests/test_agent_loop.py proves that it reproduces the reference loop's golden traces on the oracle classes;
    the GPU test then runs the restatement on the PRODUCT classes against the same golden traces.

Whatever `mem`, `net`, `buf` objects are passed in (reference files, oracle classes, product classes) are used only
through the reference's call surface (SURVEY §8b)."""
import csv
import random
import types
import zlib

import numpy as np


def loop_config(**kw):
    """The argparse fields of src/main.py:16-84 that Agent / Statistics / the epoch loop read, scaled down to a test
    (reference defaults in brackets)."""
    d = dict(random_starts=30,                 # [30]
             history_length=4, batch_size=32, screen_height=84, screen_width=84,
             exploration_rate_start=1.0,       # [1]
             exploration_rate_end=0.1,         # [0.1]
             exploration_decay_steps=400,      # [1000000]
             exploration_rate_test=0.05,       # [0.05]
             train_frequency=4,                # [4]
             train_repeat=1,                   # [1]
             target_steps=200,                 # [10000] -> every 50 updates here, 2500 in configs[2]
             start_epoch=0, epochs=2,          # [0, 200]
             random_steps=300,                 # [50000]
             train_steps=500,                  # [250000]
             test_steps=100,                   # [125000]
             replay_size=10000,                # configs[0]: replay 10k
             csv_file=None, random_seed=666,
             # network side (main.py:36-54 defaults)
             discount_rate=0.99, learning_rate=0.00025, decay_rate=0.95, clip_error=1, min_reward=-1, max_reward=1,
             batch_norm=False, optimizer="rmsprop", backend="gpu", device_id=0, datatype="float32",
             stochastic_round=False, save_weights_prefix=None)
    d.update(kw)
    return types.SimpleNamespace(**d)


class Trace:
    """What a run leaves behind: enough to tell whether two runs made the same decisions with the same numbers."""

    def __init__(self):
        self.actions, self.rewards, self.terminals, self.rates = [], [], [], []
        self.costs = []                 # cost[0,0] of every DeepQNetwork.train (callback.on_train)
        self.q_rows = []                # row 0 of every DeepQNetwork.predict, in call order
        self.stats_q = []               # positions in q_rows of the Statistics.write predicts (validation states)
        self.rng_crc = []               # crc32 of random.getstate() at every phase boundary
        self.phase_rows = []            # (epoch, phase, steps, nr_games, avg_reward, min, max, meanq, meancost, updates)
        self.mem_cursor = []            # (count, current) at every phase boundary

    def mark(self, mem):
        self.rng_crc.append(zlib.crc32(repr(random.getstate()).encode()) & 0xffffffff)
        self.mem_cursor.append((int(mem.count), int(mem.current)))

    def arrays(self):
        a = max((len(q) for q in self.q_rows), default=0)
        return dict(actions=np.array(self.actions, np.uint8), rewards=np.array(self.rewards, np.int64),
                    terminals=np.array(self.terminals, np.uint8), rates=np.array(self.rates, np.float64),
                    costs=np.array(self.costs, np.float32),
                    q_rows=np.array(self.q_rows, np.float32).reshape(len(self.q_rows), a),
                    rng_crc=np.array(self.rng_crc, np.uint32), mem_cursor=np.array(self.mem_cursor, np.int64),
                    phase_rows=np.array([[float(x) for x in r[2:]] for r in self.phase_rows], np.float64))


class RecordingNet:
    """Forwards everything to the wrapped DeepQNetwork; notes row 0 of each predict()."""

    def __init__(self, net, trace):
        object.__setattr__(self, "_net", net)
        object.__setattr__(self, "_trace", trace)

    def __getattr__(self, name):
        return getattr(self._net, name)

    def __setattr__(self, name, value):
        setattr(self._net, name, value)

    def predict(self, states):
        q = self._net.predict(states)
        self._trace.q_rows.append(np.array(q[0], np.float32))
        return q


class _Tee:
    """agent.callback / net.callback: record, then forward to the reference's Statistics object."""

    def __init__(self, stats, trace):
        self.stats, self.trace = stats, trace

    def on_step(self, action, reward, terminal, screen, exploration_rate):
        t = self.trace
        t.actions.append(int(action)); t.rewards.append(int(reward)); t.terminals.append(bool(terminal))
        t.rates.append(float(exploration_rate))
        self.stats.on_step(action, reward, terminal, screen, exploration_rate)

    def on_train(self, cost):
        self.trace.costs.append(np.float32(cost))
        self.stats.on_train(cost)


def _read_csv_rows(path):
    with open(path, newline="") as f:
        rows = list(csv.reader(f))
    return rows[1:]


def run_reference_loop(Agent, Statistics, env, mem, net, cfg, csv_path):
    """src/main.py:89-90,103-106,130-162 with the reference's own Agent and Statistics classes."""
    trace = Trace()
    cfg = types.SimpleNamespace(**vars(cfg))
    cfg.csv_file = csv_path
    if cfg.random_seed:
        random.seed(cfg.random_seed)                       # main.py:89-90
    rnet = RecordingNet(net, trace)
    agent = Agent(env, mem, rnet, cfg)                     # main.py:105
    stats = Statistics(agent, rnet, mem, env, cfg)         # main.py:106
    tee = _Tee(stats, trace)
    agent.callback = tee
    net.callback = tee
    trace.mark(mem)
    if cfg.random_steps:                                   # main.py:130-137
        env.setMode("train")
        stats.reset()
        agent.play_random(cfg.random_steps)
        stats.write(0, "random")
        trace.mark(mem)
    for epoch in range(cfg.start_epoch, cfg.epochs):       # main.py:140-162
        if cfg.train_steps:
            env.setMode("train")
            stats.reset()
            agent.train(cfg.train_steps, epoch)
            stats.write(epoch + 1, "train")
            trace.mark(mem)
        if cfg.test_steps:
            env.setMode("test")
            stats.reset()
            agent.test(cfg.test_steps, epoch)
            stats.write(epoch + 1, "test")
            trace.mark(mem)
    stats.close()
    net.callback = None
    for r in _read_csv_rows(csv_path):
        # epoch, phase, steps, nr_games, average_reward, min, max, last_eps, total_train_steps, replay_count, meanq,
        # meancost, weight_updates, ...
        trace.phase_rows.append((r[0], r[1], r[2], r[3], r[4], r[5], r[6], r[10], r[11], r[12]))
    return trace


# ------------------------------------------------------------------------------------------------------------
# Independent restatement (this repository's own code).  Each block names the reference lines whose behaviour it
# reproduces; the structure is deliberately different (one flat driver, explicit state record) so that equality of
# traces with run_reference_loop is a real check, not a tautology.
# ------------------------------------------------------------------------------------------------------------
def run_restated_loop(env, mem, net, buf, cfg, fused_train=None):
    """`fused_train(mem, net, repeat, epoch)` may replace the `train_repeat` x (getMinibatch, train) pair of
    agent.py:110-114 with a fused equivalent (the product's one-call path); default is the reference's two calls."""
    trace = Trace()
    if cfg.random_seed:
        random.seed(cfg.random_seed)
    rnet = RecordingNet(net, trace)
    n_actions = env.numActions()
    S = types.SimpleNamespace(total_train_steps=cfg.start_epoch * cfg.train_steps,      # agent.py:21
                              validation=None, steps=0, games=0, game_reward=0, avg_reward=0.0,
                              lo=None, hi=None, avg_cost=0.0)

    class _Hooks:        # net.callback target: statistics.py:70-71 running mean over ALL weight updates
        @staticmethod
        def on_train(cost):
            trace.costs.append(np.float32(cost))
            S.avg_cost += (cost - S.avg_cost) / net.train_iterations
    net.callback = _Hooks

    def new_phase():      # statistics.py:46-56
        S.steps = S.games = 0
        S.game_reward = 0
        S.avg_reward = 0.0
        S.lo, S.hi = None, None
        S.avg_cost = 0.0

    def random_restart():  # agent.py:29-39
        env.restart()
        for _ in range(random.randint(cfg.history_length, cfg.random_starts) + 1):
            env.act(0)
            if env.isTerminal():
                env.restart()
            buf.add(env.getScreen())

    def one_step(eps):     # agent.py:48-85 + statistics.py:58-68
        if random.random() < eps:
            action = random.randrange(n_actions)
        else:
            action = int(np.argmax(rnet.predict(buf.getStateMinibatch())[0]))
        reward = env.act(action)
        screen = env.getScreen()
        terminal = env.isTerminal()
        buf.add(screen)
        if terminal:
            random_restart()
        trace.actions.append(int(action)); trace.rewards.append(int(reward)); trace.terminals.append(bool(terminal))
        trace.rates.append(float(eps))
        S.game_reward += reward
        S.steps += 1
        if terminal:
            S.games += 1
            S.avg_reward += float(S.game_reward - S.avg_reward) / S.games
            S.lo = S.game_reward if S.lo is None else min(S.lo, S.game_reward)
            S.hi = S.game_reward if S.hi is None else max(S.hi, S.game_reward)
            S.game_reward = 0
        return action, reward, screen, terminal

    def end_phase(epoch, phase):   # statistics.py:73-120 (csv enabled)
        if S.games == 0:
            S.games, S.avg_reward = 1, S.game_reward
        if S.validation is None and mem.count > mem.batch_size:
            S.validation = mem.getMinibatch()[0]           # the persistent prestates buffer, aliased (SURVEY §3.5)
        if S.validation is not None:
            trace.stats_q.append(len(trace.q_rows))
        meanq = float(np.mean(np.max(rnet.predict(S.validation), axis=1))) if S.validation is not None else 0
        import sys
        lo = sys.maxsize if S.lo is None else S.lo
        hi = -sys.maxsize - 1 if S.hi is None else S.hi
        trace.phase_rows.append((epoch, phase, S.steps, S.games, S.avg_reward, lo, hi, meanq, S.avg_cost,
                                 net.train_iterations))
        trace.mark(mem)

    def eps_now():                 # agent.py:41-46
        if S.total_train_steps < cfg.exploration_decay_steps:
            return cfg.exploration_rate_start - S.total_train_steps * \
                (cfg.exploration_rate_start - cfg.exploration_rate_end) / cfg.exploration_decay_steps
        return cfg.exploration_rate_end

    trace.mark(mem)
    if cfg.random_steps:           # main.py:130-137, agent.py:87-94
        env.setMode("train")
        new_phase()
        env.restart()
        for _ in range(cfg.random_steps):
            mem.add(*one_step(1))
        end_phase(0, "random")
    for epoch in range(cfg.start_epoch, cfg.epochs):
        if cfg.train_steps:        # main.py:143-149, agent.py:96-116
            env.setMode("train")
            new_phase()
            for i in range(cfg.train_steps):
                mem.add(*one_step(eps_now()))
                if cfg.target_steps and i % cfg.target_steps == 0:
                    net.update_target_network()
                if mem.count > mem.batch_size and i % cfg.train_frequency == 0:
                    if fused_train is not None:
                        fused_train(mem, net, cfg.train_repeat, epoch)
                    else:
                        for _ in range(cfg.train_repeat):
                            net.train(mem.getMinibatch(), epoch)
                S.total_train_steps += 1
            end_phase(epoch + 1, "train")
        if cfg.test_steps:         # main.py:156-162, agent.py:118-124
            env.setMode("test")
            new_phase()
            random_restart()
            for _ in range(cfg.test_steps):
                one_step(cfg.exploration_rate_test)
            end_phase(epoch + 1, "test")
    net.callback = None
    return trace


# ------------------------------------------------------------------------------------------------------------
# Oracle-side classes with the reference's call surface (the checker; never the product)
# ------------------------------------------------------------------------------------------------------------
def oracle_classes():
    from oracle import dqn_oracle as O
    from oracle.mt19937 import MT19937
    from oracle.replay_oracle import ReplayOracle, StateBufferOracle

    class OracleReplayMemory(ReplayOracle):
        """ReplayOracle drawing from the process-global `random`, like src/replay_memory.py:59."""

        def __init__(self, size, args):
            super().__init__(size, args.screen_height, args.screen_width, args.history_length, args.batch_size)

        def getMinibatch(self):
            rng = MT19937.from_python(random)
            out = ReplayOracle.getMinibatch(self, rng)
            rng.to_python(random)
            return out

    class OracleStateBuffer(StateBufferOracle):
        def __init__(self, args):
            super().__init__(args.screen_height, args.screen_width, args.history_length, args.batch_size)

    class OracleDeepQNetwork(O.DQNOracle):
        def __init__(self, num_actions, args):
            super().__init__(num_actions, batch_size=args.batch_size, discount_rate=args.discount_rate,
                             learning_rate=args.learning_rate, decay_rate=args.decay_rate,
                             clip_error=args.clip_error, min_reward=args.min_reward, max_reward=args.max_reward,
                             target_steps=args.target_steps, optimizer=getattr(args, "optimizer", "rmsprop"),
                             weights=O.xavier_init(num_actions, args.random_seed))
            # deepqnetwork.py:63-70 initialises a separate target model; it is overwritten by the first
            # update_target_network (agent.py:105 at i == 0) before anything reads it, so a copy is equivalent.

    return OracleReplayMemory, OracleStateBuffer, OracleDeepQNetwork


class LockstepNet:
    """Runs a SUBJECT DeepQNetwork (the product) and a CHECKER (the numpy oracle) side by side behind one
    DeepQNetwork call surface, inside the real control loop.

    DQN + RMSProp on a fresh network is chaotic in fp32 (two CPU implementations of the same algorithm disagree on
    a third of the greedy actions after ~20 updates — tests/test_gpu_net.py::test_trajectory_20_steps…), so whole-run
    trace equality between ANY two implementations is not a meaningful bar.  Instead every call is compared where
    it happens, and the subject's parameters are re-based on the checker's every `resync` updates so that what is
    measured is `resync` consecutive product updates from a common starting point — along the trajectory the
    reference loop actually visits (replay contents, target syncs, ε schedule), not on hand-made minibatches.
    The loop itself follows the SUBJECT's decisions."""

    def __init__(self, subject, checker, resync=4):
        self.subject, self.checker, self.resync = subject, checker, resync
        self.batch_size = subject.batch_size
        self.callback = None
        self.since_sync = 0
        self.cost_err = []          # (updates since re-base, |cost - ref| / |ref|)
        self.q_err = []             # (updates since re-base, max|dQ| / max|Q|) per predict
        self.ties = []              # (predict index, relative top-2 gap, q error) where the greedy actions differ
        self.predicts = 0

    @property
    def train_iterations(self):
        return self.subject.train_iterations

    def update_target_network(self):
        self.subject.update_target_network()
        self.checker.update_target_network()

    def predict(self, states):
        q = self.subject.predict(states)
        ref = self.checker.predict(np.asarray(states))
        scale = max(float(np.abs(ref).max()), 1e-30)
        self.q_err.append((self.since_sync, float(np.abs(q - ref).max()) / scale))
        if int(np.argmax(q[0])) != int(np.argmax(ref[0])):
            s = np.sort(ref[0])
            self.ties.append((self.predicts, float(s[-1] - s[-2]) / max(float(np.abs(ref[0]).max()), 1e-30),
                              float(np.abs(q[0] - ref[0]).max()) / max(float(np.abs(ref[0]).max()), 1e-30)))
        self.predicts += 1
        return q

    def train(self, minibatch, epoch):
        box = []
        self.subject.callback = types.SimpleNamespace(on_train=box.append)
        self.subject.train(minibatch, epoch)            # first: a pristine device handle is trained in place from the ring
        self.subject.callback = None
        pre, act, rew, post, term = minibatch           # now materialise it: the checker needs host copies
        host = (np.array(pre), np.array(act), np.array(rew), np.array(post), np.array(term))
        ref = float(self.checker.train(host, epoch))
        self.since_sync += 1
        self.cost_err.append((self.since_sync, abs(float(box[0]) - ref) / max(abs(ref), 1e-30)))
        if self.since_sync >= self.resync:
            self.rebase()
        if self.callback:
            self.callback.on_train(box[0])

    def rebase(self):
        self.subject.set_weights(self.checker.weights, self.checker.states)
        if self.checker.target_weights is not self.checker.weights:      # the target copy was taken from drifted weights
            self.subject.set_weights(self.checker.target_weights, None, which=1)
        self.since_sync = 0
