"""Agent: the A3C worker loop (reference src/agent.py:14-396: before_train / train / predict /
observe / batch_update / lr), batched over ``num_envs`` environments per GPU.

What maps to what (DESIGN.md has the full table):
  predict      agent.py:141-151   forward of the current stack + action selection (sampled from
                                  pi, network.py:72, instead of the epsilon-greedy of the async-Q code)
  observe      agent.py:153-167   reward clip (in-kernel), history push (K1 fused), rollout append,
                                  update every t_max steps (reference: every train_frequency)
  batch_update agent.py:169-207   bootstrap, n-step returns, loss grads, backward, [allreduce],
                                  clip + RMSProp  == Algorithm 3's accumulate-then-apply
  lr           agent.py:393-395   linear anneal on the worker-local step

Asynchronous hogwild updates through a parameter server (main.py:60-62, agent.py:321) become
synchronous data parallelism: every rank holds a replica, gradients are summed with one NCCL
all-reduce per t_max cycle, every rank applies the identical update.
"""
import json
import os

import torch
import torch.distributed as dist

from .. import _cabi
from .base import BaseModel
from .history import History
from .network import make_network


class Agent(BaseModel):
    def __init__(self, config, environment, optimizer=None, lr_op=None, device=None):
        super(Agent, self).__init__(config)
        self.weight_dir = 'weights'
        self.env = environment
        self.device = torch.device(device if device is not None else environment.device)
        self.history = History(self.config, num_envs=self.num_envs, device=self.device)

        self.rank = dist.get_rank() if dist.is_available() and dist.is_initialized() else 0
        self.world_size = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
        self.env_id_base = self.rank * self.num_envs           # global env ids: sharding-independent RNG
        self.global_envs = self.world_size * self.num_envs

        self.step_op = 0                                         # agent.py:25 global step (host int)
        # config.py:36 dueling: Wang et al. 2016's dueling Q heads for the Q learners (Network.dueling);
        # a policy/value network has no dueling form
        self.dueling = bool(getattr(config, 'dueling', False))
        if self.dueling and getattr(config, 'loss_mode', 'a3c') == 'a3c':
            raise ValueError("dueling=True needs a Q learner (loss_mode 'async_q', 'nstep_q' or 'sarsa'); "
                             "loss_mode 'a3c' trains a policy/value network, which has no dueling form")
        # config.py dueling_streams: the dueling architecture with a hidden layer per stream
        # (Network.dueling_streams), an option of the dueling heads
        self.dueling_streams = bool(getattr(config, 'dueling_streams', False))
        if self.dueling_streams and getattr(config, 'loss_mode', 'a3c') == 'a3c':
            raise ValueError("dueling_streams=True needs a Q learner (loss_mode 'async_q', 'nstep_q' or 'sarsa'); "
                             "loss_mode 'a3c' trains a policy/value network, which has no dueling form")
        if self.dueling_streams and not self.dueling:
            raise ValueError("dueling_streams=True gives the dueling heads a hidden layer per stream; it needs "
                             "dueling=True")
        # config.py:35 double_q: Double DQN targets (van Hasselt et al. 2016) for the learners that
        # bootstrap from a max; a3c has no max to decouple, sarsa bootstraps from the action taken in s'
        self.double_q = bool(getattr(config, 'double_q', False))
        if self.double_q and getattr(config, 'loss_mode', 'a3c') not in ('async_q', 'nstep_q'):
            raise ValueError("double_q=True needs a learner that bootstraps from max_a Q (loss_mode 'async_q' or "
                             "'nstep_q'); loss_mode %r has no max to decouple"
                             % (getattr(config, 'loss_mode', 'a3c'),))
        # config.py lstm: Mnih et al. 2016's A3C LSTM agent (Network.lstm), a policy/value network
        self.lstm = bool(getattr(config, 'lstm', False))
        if self.lstm and getattr(config, 'loss_mode', 'a3c') != 'a3c':
            raise ValueError("lstm=True is the A3C LSTM agent (loss_mode 'a3c'); loss_mode %r has no recurrent form"
                             % (getattr(config, 'loss_mode', 'a3c'),))
        # network.py:30-55: 'nips' (what agent.py:226-252 wires, the default) or 'nature'
        self.network = make_network(
            DQN_type=getattr(config, 'DQN_type', 'nips'), action_size=self.env.action_size, data_format=self.cnn_format,
            history_length=self.history_length, screen_height=self.screen_height,
            screen_width=self.screen_width, gamma=self.discount, beta=self.beta,
            num_envs=self.num_envs, t_max=self.t_max, device=self.device, seed=self.seed,
            decay=self.decay, epsilon=self.epsilon, clip_norm=self.clip_norm,
            min_reward=self.min_reward, max_reward=self.max_reward, dueling=self.dueling, double_q=self.double_q,
            dueling_streams=self.dueling_streams, lstm=self.lstm)
        self.w = self.network.w
        # the per-cycle exchange runs inside the library (arl_comm_init / arl_backward(allreduce=1):
        # NCCL, bucketed so that the fc256 gradient travels while the conv backward kernels run);
        # collective='torch' keeps the all-reduce in torch.distributed (debugging / gloo)
        # 'p2p': no collective kernel at all -- every rank reads the others' gradients over NVLink
        # peer memory inside the norm pass of the update (arl_exchange_clip_rmsprop)
        # 'auto' (default): 'p2p' on 2 GPUs, 'library' beyond -- measured (profiles/r02_exchange.txt):
        # the one-shot peer read wins by 8 us per cycle at N=2 and loses 33 us at N=8, where every
        # rank pulls 7 x 2.7 MB while NCCL reduces inside the NVSwitch (NVLS)
        self.collective = getattr(config, 'collective', 'auto')
        if self.collective == 'auto':
            self.collective = 'p2p' if self.world_size == 2 else 'library'
        if self.collective not in ('p2p', 'library', 'torch'):
            raise ValueError("collective must be 'auto', 'p2p', 'library' or 'torch'")
        if self.world_size > 1 and self.collective in ('p2p', 'library'):
            _cabi.comm_init(self.device)
            if self.collective == 'p2p':
                with torch.cuda.device(self.device):
                    _cabi.call("arl_comm_enable_p2p", int(self.network.params.numel()))

        T, B = self.t_max, self.num_envs
        self.batch_reward = torch.zeros(T, B, device=self.device)
        self.batch_terminal = torch.zeros(T, B, dtype=torch.uint8, device=self.device)
        self.t = 0                                               # position inside the rollout
        self.step = 0
        self.T = 0
        self.update_count = 0
        # loss_mode 'async_q' = the learner the reference actually runs (SURVEY D1): Q head,
        # epsilon-greedy, 1-step targets from a target network (agent.py:141-207, 298-314)
        # loss_mode 'nstep_q' = the paper's asynchronous n-step Q-learning: the same Q head,
        # epsilon-greedy schedule and target network, n-step returns bootstrapped from
        # max_a Q(s_T; theta^-) -- the A3C cycle with another loss kernel, on the graph-replayed path
        # loss_mode 'sarsa' = the paper's asynchronous one-step Sarsa: async_q's 1-step targets with
        # Q(s', a'; theta^-) of the action a' actually taken in s'; on the graph-replayed path too
        self.loss_mode = getattr(config, 'loss_mode', 'a3c')
        if self.loss_mode not in ('a3c', 'async_q', 'nstep_q', 'sarsa'):
            raise ValueError("loss_mode must be 'a3c', 'async_q', 'nstep_q' or 'sarsa', got %r" % (self.loss_mode,))
        self.has_target = self.loss_mode in ('async_q', 'nstep_q', 'sarsa')
        if self.has_target:
            self.network.make_target(one_step=self.loss_mode != 'nstep_q', next_actions=self.loss_mode == 'sarsa')
            self._last_target_sync = 0
        # sarsa: the update drew a_T, the action the next rollout's step 0 takes (row T of
        # network.sarsa_actions); False before the first update and after before_train
        self.sarsa_pending = False
        self.batch_action = self.network.sampled_action.view(T, B)
        # CUDA graphs of the loop (SURVEY a16): the device work of ``predict`` and of ``observe``
        # (+ the learner step at the end of a rollout) is captured once per distinct set of launch
        # arguments -- rollout slot, ring position, frame / reward buffers -- and replayed from then
        # on.  The two host values that change on every step, the Philox step and the step the
        # learning rate is annealed on, are read from ``step_dev`` (device memory) instead.
        self.cuda_graphs = bool(getattr(config, 'cuda_graphs', True)) and self.loss_mode in ('a3c', 'nstep_q', 'sarsa')
        self.max_graphs = int(getattr(config, 'max_graphs', 1024))
        self.graph_warmup_updates = 2                            # eager cycles first (lazy init, autotune)
        self.step_dev = torch.zeros(1, dtype=torch.int64, device=self.device)
        self._step_dev_host = None                               # value step_dev holds, if known
        self._graphs = {}
        self._graph_pool = None
        self.graph_replays = 0
        self.graph_kernels_replayed = 0                          # library kernels launched by replays

    # -- agent.py:33-50 ---------------------------------------------------------------------
    def before_train(self, is_chief=True):
        self.step = self.step_op
        self.T = self.step_op * self.global_envs                 # agent.py:165 counts every worker's frames
        self.env.new_random_game()
        # agent.py:37-38: the stack starts as 4 copies of the first screen (K1, replicate=4)
        self.history.add(self.env.frames, replicate=self.history_length)
        self.t = 0
        self.network.reset_lstm_state()                          # every game starts over: (h, c) = 0
        self.update_target_q_network()                           # main.py:92
        if self.has_target:
            self._last_target_sync = self.T
        self.sarsa_pending = False                               # the first step draws its action
        return self.env.frames, 0, 0, self.env.terminal, range(self.step, self.max_step)

    # -- agent.py:52-67 ---------------------------------------------------------------------
    def train(self, sv=None, is_chief=True, num_steps=None):
        screen, reward, action, terminal, iterator = self.before_train(is_chief)
        end = self.max_step if num_steps is None else min(self.max_step, self.step + num_steps)
        ran = False
        for self.step in range(self.step, end):
            # 1. predict
            action = self.predict()
            # 2. act
            screen, reward, terminal = self.env.act(action, is_training=True, fused=True)
            # 3. observe
            self.observe(screen, reward, action, terminal)
            # agent.py:66-67: the envs that died restart (their own random-start draw each); like
            # the reference, the History is NOT reset on terminal and the restart screen is dropped
            if self.env.per_env_restart:
                self.env.new_random_game(mask=terminal)
            ran = True
        if ran:
            self.step_op = self.step + 1
        return self.step_op

    # -- agent.py:69-139 --------------------------------------------------------------------
    def train_with_summary(self, sv=None, is_chief=True, num_steps=None, log_path=None):
        """The chief's loop (agent.py:69-139): same steps as ``train`` plus the statistics the
        reference injects every ``test_step`` steps, with the reference's tag names, as JSON lines
        (``log_path``) instead of TF summaries.  The running sums live on the device; one small
        device->host read per ``test_step`` window."""
        screen, reward, action, terminal, iterator = self.before_train(is_chief)
        end = self.max_step if num_steps is None else min(self.max_step, self.step + num_steps)
        dev, B = self.device, self.num_envs
        zeros = lambda *shape: torch.zeros(*shape, device=dev)
        ep_reward = zeros(B)                                     # agent.py:72 per env
        # [sum reward, #games, sum/max/min episode reward, sum loss, sum q]
        acc = dict(reward=zeros(()), games=zeros(()), ep_sum=zeros(()),
                   ep_max=torch.full((), -float('inf'), device=dev),
                   ep_min=torch.full((), float('inf'), device=dev), loss=zeros(()), q=zeros(()))
        action_hist = torch.zeros(self.env.action_size, device=dev)
        updates = 0
        test_step = max(1, int(self.test_step))
        records = []
        out = open(log_path, 'a') if (log_path and is_chief) else None
        ran = False
        for self.step in range(self.step, end):
            ran = True
            action = self.predict()
            screen, reward, terminal = self.env.act(action, is_training=True, fused=True)
            before = self.update_count
            self.observe(screen, reward, action, terminal, is_chief=True)
            if self.env.per_env_restart:                         # agent.py:66-67
                self.env.new_random_game(mask=terminal)
            if self.update_count != before:                      # agent.py:199-201
                sums = self.network.loss_sums
                if self.has_target:                              # async_q, nstep_q, sarsa: {sum delta^2, sum Q}
                    n = float(self.t_max * B)
                    acc['loss'] += sums[0] / n
                    acc['q'] += sums[1] / n
                else:
                    acc['loss'] += (sums[0] + sums[1]) / float(B)
                    acc['q'] += self.network.value.mean()
                updates += 1
            term = terminal.bool()
            r = torch.clamp(reward, self.min_reward, self.max_reward)   # observe clips (agent.py:154)
            finished = torch.where(term, ep_reward, torch.zeros_like(ep_reward))
            acc['games'] += term.sum()
            acc['ep_sum'] += finished.sum()
            acc['ep_max'] = torch.maximum(acc['ep_max'], torch.where(
                term, ep_reward, torch.full_like(ep_reward, -float('inf'))).max())
            acc['ep_min'] = torch.minimum(acc['ep_min'], torch.where(
                term, ep_reward, torch.full_like(ep_reward, float('inf'))).min())
            ep_reward = torch.where(term, torch.zeros_like(ep_reward), ep_reward + r)   # agent.py:97-102
            acc['reward'] += r.sum()
            action_hist += torch.bincount(action.long(), minlength=self.env.action_size).float()
            if self.step % test_step == test_step - 1:           # agent.py:104
                vals = {k: float(v) for k, v in acc.items()}
                games = int(vals['games'])
                rec = {
                    'step': self.step, 'T': self.T,
                    'average.reward': vals['reward'] / (test_step * B),
                    'average.loss': vals['loss'] / max(updates, 1),
                    'average.q': vals['q'] / max(updates, 1),
                    'episode.max reward': vals['ep_max'] if games else 0.0,
                    'episode.min reward': vals['ep_min'] if games else 0.0,
                    'episode.avg reward': vals['ep_sum'] / games if games else 0.0,
                    'episode.num of game': games,
                    'episode.actions': [int(c) for c in action_hist.tolist()],
                    'training.learning_rate': self.lr,
                }
                records.append(rec)
                if out is not None:
                    out.write(json.dumps(rec) + "\n")
                    out.flush()
                for k, v in acc.items():                          # agent.py:133-139
                    v.fill_(-float('inf') if k == 'ep_max' else float('inf') if k == 'ep_min' else 0.0)
                action_hist.zero_()
                updates = 0
        if out is not None:
            out.close()
        if ran:
            self.step_op = self.step + 1
        return records

    # -- checkpoints: agent.py:29 Saver(w + step_op), main.py:74-80 Supervisor autosave ------
    def save_checkpoint(self, checkpoint_dir=None):
        """Weights under the reference's variable names + the RMSProp slot (which the reference
        forgets to save) + the step counter (agent.py:25, 34)."""
        d = checkpoint_dir or self.checkpoint_dir
        path = self.network.save_model(checkpoint_dir=d, step=self.step_op)
        if self.loss_mode == 'async_q':
            torch.save(self.network.target_params.cpu(), os.path.join(d, "target-%d.pt" % self.step_op))
        elif self.loss_mode == 'nstep_q':                         # + where the sync schedule stands
            torch.save({"target": self.network.target_params.cpu(), "last_target_sync": self._last_target_sync},
                       os.path.join(d, "target-%d.pt" % self.step_op))
        elif self.loss_mode == 'sarsa':                           # + the action a_T the next step takes
            net = self.network
            torch.save({"target": net.target_params.cpu(), "last_target_sync": self._last_target_sync,
                        "pending_action": net.sarsa_actions[net.t_max * net.num_envs:].cpu(),
                        "pending": self.sarsa_pending},
                       os.path.join(d, "target-%d.pt" % self.step_op))
        return path

    def load_checkpoint(self, checkpoint_dir=None):
        """Resume (agent.py:34 ``self.step = self.step_op.eval()``).  Returns True if restored."""
        d = checkpoint_dir or self.checkpoint_dir
        if not self.network.load_model(checkpoint_dir=d):
            return False
        self.step_op = self.network.loaded_step
        if self.has_target:
            p = os.path.join(d, "target-%d.pt" % self.step_op)
            if os.path.exists(p):
                saved = torch.load(p)
                if isinstance(saved, dict):                      # nstep_q, sarsa
                    self._last_target_sync = int(saved["last_target_sync"])
                    if "pending" in saved:                       # sarsa
                        net = self.network
                        net.sarsa_actions[net.t_max * net.num_envs:].copy_(saved["pending_action"].to(self.device))
                        self.sarsa_pending = bool(saved["pending"])
                    saved = saved["target"]
                self.network.target_params.copy_(saved.to(self.device))
            else:
                self.network.update_target()
        return True

    # -- CUDA-graph plumbing ----------------------------------------------------------------
    def _graphs_on(self):
        return (self.cuda_graphs and self.network.timed is None
                and self.update_count >= self.graph_warmup_updates
                and (self.world_size == 1 or self.collective in ('p2p', 'library')))

    def _sync_step_dev(self):
        """``step_dev`` mirrors the host's ``self.step``; callers that move ``self.step`` by hand
        (tests drive the loop manually) are followed with one fill."""
        if self._step_dev_host != self.step:
            self.step_dev.fill_(int(self.step))
            self._step_dev_host = self.step

    def _run(self, key, launches):
        """Run ``launches`` (device work only, no host state) -- replaying its captured graph when
        one exists for ``key``, capturing it on first sight."""
        if not self._graphs_on():
            launches()
            return
        g = self._graphs.get(key)
        if g is None:
            if len(self._graphs) >= self.max_graphs:
                launches()
                return
            if self._graph_pool is None:
                self._graph_pool = torch.cuda.graph_pool_handle()
            graph = torch.cuda.CUDAGraph()
            n0 = _cabi.launch_count()
            with torch.cuda.graph(graph, pool=self._graph_pool):
                launches()
            g = self._graphs[key] = (graph, _cabi.launch_count() - n0)   # + its kernel-node count
        g[0].replay()
        self.graph_replays += 1
        self.graph_kernels_replayed += g[1]

    # -- agent.py:141-151 -------------------------------------------------------------------
    def predict(self, s_t=None, test_ep=None):
        """Forward of the current stack (already in the ring; ``s_t`` is accepted for signature
        compatibility and ignored) and one sampled action per env."""
        net, t = self.network, self.t
        if self.loss_mode == 'async_q':                          # agent.py:142-149
            net.forward(self.history, t)
            ep = self.ep if test_ep is None else test_ep
            return net.egreedy(t, self.step, self.seed, ep, self.env_id_base)
        if self.loss_mode in ('nstep_q', 'sarsa') and test_ep is not None:   # a fixed epsilon: eager
            return net.forward_egreedy(self.history, t, self.seed, self.env_id_base, step=self.step, ep=test_ep)
        self._sync_step_dev()
        refresh = net._fc_w_stale()
        # sarsa: step 0 after an update takes the action a_T that update drew (Mnih et al. 2016:
        # choose a', accumulate, update, take a'); the forward still runs, its activations are s_0's
        take_pending = self.loss_mode == 'sarsa' and t == 0 and self.sarsa_pending

        def launches():                                        # forward + heads + Philox draw
            if take_pending:
                r = net._rows(0)
                net.forward(self.history, 0, refresh=refresh)
                net.sampled_action[r].copy_(net.sarsa_actions[self.t_max * self.num_envs:])   # cudaMemcpyAsync
            elif self.loss_mode in ('nstep_q', 'sarsa'):       # agent.py:142-149, epsilon from step_dev
                net.forward_egreedy(self.history, t, self.seed, self.env_id_base, step_dev=self.step_dev,
                                    ep_sched=self._ep_sched(), refresh=refresh)
            else:
                net.forward_sample(self.history, t, 0, self.seed, self.env_id_base, step_dev=self.step_dev,
                                   refresh=refresh, **self._lstm_reset(t))
        self._run(('predict', t, self.history.head, refresh, take_pending), launches)
        return net.sampled_action[net._rows(t)]

    def _lstm_reset(self, t):
        """The ``reset`` argument of the LSTM forward entering rollout step ``t`` (none without an LSTM): the
        terminal row of step t-1, for step 0 the previous rollout's last (a fixed row: the graph key t covers it)."""
        return dict(reset=self.batch_terminal[(t - 1) % self.t_max]) if self.lstm else {}

    def _ep_sched(self):
        """agent.py:142-144's constants, for the epsilon the kernels evaluate from ``step_dev``."""
        return (self.ep_start, self.ep_end, self.ep_end_t, self.learn_start)

    # -- agent.py:351-391 -------------------------------------------------------------------
    def play(self, sv=None, is_chief=True, n_step=10000, n_episode=100, test_ep=None, render=False):
        """Evaluation episodes (agent.py:351-391) on all ``num_envs`` environments at once: a fresh
        History seeded with 4 copies of the first screen (agent.py:365-366), then predict / act
        (is_training=False: no life-loss terminal) / add until every env has finished its episode
        or ``n_step`` steps have passed.  Action selection: epsilon-greedy with ``test_ep``
        (default ep_end, agent.py:352-353) in async_q / nstep_q / sarsa mode, a sample from the policy
        in a3c mode.
        Returns (best_reward, best_idx, per-episode mean reward over the envs); gym's monitor
        (agent.py:357-359) is the emulator's business and not reproduced."""
        if test_ep is None:
            test_ep = self.ep_end
        test_history = History(self.config, num_envs=self.num_envs, device=self.device)
        best_reward, best_idx, means = 0.0, 0, []
        step = 0
        for idx in range(int(n_episode)):
            self.env.new_random_game()
            test_history.add(self.env.frames, replicate=self.history_length)
            self.network.reset_lstm_state(play=True)
            current = torch.zeros(self.num_envs, device=self.device)
            alive = torch.ones(self.num_envs, dtype=torch.bool, device=self.device)
            for _ in range(int(n_step)):
                # 1. predict   2. act   3. observe
                action = self.network.evaluate(test_history, step, self.seed + 1,
                                               ep=test_ep if self.has_target else None,
                                               env_id_base=self.env_id_base)
                screen, reward, terminal = self.env.act(action, is_training=False, fused=True)
                test_history.add(screen)
                current += torch.where(alive, reward, torch.zeros_like(reward))
                alive &= ~terminal.bool()
                step += 1
                if render:
                    self.env.render()
                if not bool(alive.any()):
                    break
            top = float(current.max())
            means.append(float(current.mean()))
            if top > best_reward:
                best_reward, best_idx = top, idx
        return best_reward, best_idx, means

    # -- agent.py:153-167 -------------------------------------------------------------------
    def observe(self, screen, reward, action, terminal, is_chief=False):
        fast = (reward.dtype == torch.float32 and terminal.dtype in (torch.bool, torch.uint8)
                and reward.is_contiguous() and terminal.is_contiguous())
        t, hist = self.t, self.history
        will_update = t + 1 == self.t_max                        # agent.py:162-163
        if self.loss_mode == 'async_q' or not fast:
            hist.add(screen)                                     # agent.py:156 (K1 when raw frames)
            if fast:
                _cabi.call("arl_observe_store", _cabi.ptr(reward), _cabi.ptr(terminal),
                           _cabi.ptr(self.batch_reward[t]), _cabi.ptr(self.batch_terminal[t]),
                           self.num_envs, _cabi.stream_ptr())
            else:
                self.batch_reward[t].copy_(reward)
                self.batch_terminal[t].copy_(terminal)
            self.t += 1
            if will_update:
                self.batch_update(is_chief)
        else:
            self._sync_step_dev()
            new_head = (hist.head + 1) % hist.ring_slots
            hist.head = new_head                                 # host state first: the launches read it
            refresh = self.network._fc_w_stale() if will_update else False
            # nstep_q, sarsa: rebuild the target's weight image in this update only after a target sync
            target_refresh = (self.loss_mode in ('nstep_q', 'sarsa') and will_update
                              and self.network._target_fc_w_stale())

            # bench.py: an event pair around K1 -- launched eagerly between its events, or (when the
            # events can be graph nodes) captured with the rest of the step
            k1_eager = hist.timer is not None and not hist.timer_in_graph
            if k1_eager:
                hist.push_into(screen, new_head)

            def launches():
                if not k1_eager:
                    hist.push_into(screen, new_head)             # agent.py:156: K1, fused screen + add
                # one kernel for both appends; the clip happens in K4 (agent.py:154)
                _cabi.call("arl_observe_store_advance", _cabi.ptr(reward), _cabi.ptr(terminal),
                           _cabi.ptr(self.batch_reward[t]), _cabi.ptr(self.batch_terminal[t]),
                           self.num_envs, _cabi.ptr(self.step_dev), 1, _cabi.stream_ptr())
                if will_update:
                    self._update_launches(refresh, target_refresh)
            self._run(('observe', t, new_head, screen.data_ptr(), reward.data_ptr(),
                       terminal.data_ptr(), tuple(screen.shape), will_update, refresh, k1_eager,
                       hist.timer is not None, target_refresh),
                      launches)
            self._step_dev_host = self.step + 1
            self.t += 1
            if will_update:
                self.network._param_writes += 1                  # the update wrote the parameters
                self.update_count += 1
                self.sarsa_pending = self.loss_mode == 'sarsa'
                self.t = 0
        self.T += self.global_envs                               # agent.py:165 counts every worker
        if self.has_target and self.T - self._last_target_sync >= self.target_q_update_step:
            self.update_target_q_network()                       # agent.py:166-167
            self._last_target_sync = self.T

    def _gradients(self, refresh=None, target_refresh=None):
        """The learner's gradient of the rollout (agent.py:169-207) with its scale, summed over the
        ranks when the exchange is the torch all-reduce.  ``refresh`` / ``target_refresh``: rebuild the
        prepared weight images first (None = decide from the parameter versions)."""
        net, hist = self.network, self.history
        in_lib = self.world_size > 1 and self.collective == 'library'      # the one exchange per cycle
        # a3c, nstep_q and sarsa: sum over t, mean over (global) envs (the Q learners take the A3C
        # reduction: the paper accumulates over the rollout); async_q: agent.py:312-314's mean over the
        # worker's batch
        steps = self.t_max if self.loss_mode == 'async_q' else 1
        scale = 1.0 / (steps * self.global_envs) if self.reduce_mean else 1.0 / steps
        if self.loss_mode == 'async_q':
            net.compute_q_gradients(hist, self.batch_reward, self.batch_terminal, scale, allreduce=in_lib)
        elif self.loss_mode == 'nstep_q':
            net.compute_nstep_q_gradients(hist, self.batch_reward, self.batch_terminal, scale, allreduce=in_lib,
                                          target_refresh=target_refresh, refresh=refresh)
        elif self.loss_mode == 'sarsa':                                  # a_T: step and epsilon of step_dev
            net.compute_sarsa_gradients(hist, self.batch_reward, self.batch_terminal, scale, self.step_dev,
                                        self.seed, self._ep_sched(), self.env_id_base, allreduce=in_lib,
                                        target_refresh=target_refresh, refresh=refresh)
        else:
            v_boot = net.bootstrap_value(hist, refresh=refresh,          # R = V(s_T), masked if terminal
                                         **self._lstm_reset(self.t_max))
            net.compute_gradients(hist, self.batch_reward, self.batch_terminal, v_boot, grad_scale=scale,
                                  allreduce=in_lib, refresh=False)
        if self.world_size > 1 and self.collective == 'torch':
            dist.all_reduce(net.grads, op=dist.ReduceOp.SUM)

    def _update_launches(self, refresh, target_refresh=False):
        """Device work of ``batch_update`` in a3c / nstep_q / sarsa mode with the learning rate taken from
        the device step counter (already advanced past the last frame of the rollout: offset -t_max
        gives the step of the rollout's first frame, SURVEY §8 step 9)."""
        self._gradients(refresh, target_refresh)
        self.network.apply_gradients_sched(self.step_dev, -self.t_max, self.learning_rate, self.max_step,
                                           count_write=False,
                                           exchange=self.world_size > 1 and self.collective == 'p2p')

    # -- agent.py:169-207 -------------------------------------------------------------------
    def batch_update(self, is_chief=False):
        if self.loss_mode == 'sarsa':
            # a_T is drawn with the step of the next rollout's first frame, as on the replayed path
            # (observe has advanced step_dev past this rollout's last frame there)
            self.step_dev.fill_(int(self.step) + 1)
            self._step_dev_host = self.step + 1
        self._gradients()
        self.network.apply_gradients(self.lr, exchange=self.world_size > 1 and self.collective == 'p2p')
        self.update_count += 1
        self.sarsa_pending = self.loss_mode == 'sarsa'
        self.t = 0

    def update_target_q_network(self):
        """agent.py:342-344 (async_q / nstep_q / sarsa mode; the A3C path has no target network).  A
        host copy outside the captured graphs; in nstep_q and sarsa mode the next update then rebuilds
        the target's weight image (Network._target_fc_w_stale)."""
        if self.has_target:
            self.network.update_target()

    @property
    def ep(self):
        """agent.py:142-144."""
        return self.ep_end + max(0., (self.ep_start - self.ep_end) *
                                 (self.ep_end_t - max(0., self.step - self.learn_start)) / self.ep_end_t)

    @property
    def lr(self):
        """agent.py:393-395, with ``step`` = env steps taken per env at the START of the cycle
        (SURVEY §8 step 9)."""
        step = self.step - (self.t_max - 1)
        return (self.max_step - step + 1.) / self.max_step * self.learning_rate
