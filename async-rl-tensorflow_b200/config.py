"""Hyper-parameters.  Same class names, attribute names and defaults as the
reference's config.py:1-66; the additions (t_max, num_envs, seed, reduce_mean,
resize) have no reference equivalent (SURVEY.md D4) and are marked NEW."""


class AgentConfig(object):
    scale = 10000
    display = False

    max_step = 8000 * scale              # config.py:5

    random_start = 30
    cnn_format = 'NHWC'                  # main.py:45 forces NHWC on every run
    discount = 0.99
    target_q_update_step = 4 * scale
    learning_rate = 0.0007

    decay = 0.99
    epsilon = 0.1
    momentum = 0.0
    beta = 0.01

    ep_end = 0.1
    ep_start = 1.
    ep_end_t = 400 * scale

    history_length = 4
    batch_size = 32
    train_frequency = batch_size
    learn_start = batch_size

    min_delta = -1
    max_delta = 1

    double_q = False                     # double Q-learning targets (van Hasselt et al. 2016, Double DQN) for the
                                         # learners that bootstrap from a max (async_q, nstep_q): the online network
                                         # picks a* = argmax_a Q(s'; theta), the target network evaluates
                                         # Q(s', a*; theta^-); a3c and sarsa refuse it, as does the nature trunk
    dueling = False                      # dueling Q heads (Wang et al. 2016, "average" aggregator) for the
                                         # Q learners (async_q, nstep_q, sarsa) on the nips trunk: p_w/p_b is the
                                         # advantage stream, q_w/q_b the value stream, both on fc256's output
                                         # (no hidden layer per stream); a3c refuses it
    lstm = False                         # a3c only: Mnih et al. 2016's A3C LSTM agent, 256 LSTM cells between fc256
                                         # and the heads (lstm_w/lstm_b), stepped in the rollout and trained by
                                         # truncated BPTT over t_max steps; Q learners and the nature trunk refuse it
    dueling_streams = False              # with dueling: Wang et al.'s dueling architecture, each stream on its own
                                         # 256-wide hidden layer on conv2's output (value: l4_w/l4_b, advantage:
                                         # la_w/la_b); needs dueling=True, a3c and the nature trunk refuse it

    _test_step = 0.5 * scale

    # NEW (no reference counterpart; Algorithm 3 of assets/a3c.png names t_max)
    t_max = 5                            # rollout length per update
    num_envs = 256                       # environments per process (= per GPU)
    seed = 123                           # main.py:35 random_seed default
    reduce_mean = True                   # sum over t, mean over envs (False: pure sum)
    clip_norm = 40.0                     # agent.py:319
    resize = 'cv2'                       # environment.py:5-12 executed branch
    loss_mode = 'a3c'                    # 'a3c' (network.py heads/loss) | 'async_q' (agent.py as run) |
                                         # 'nstep_q' (the paper's asynchronous n-step Q-learning) |
                                         # 'sarsa' (the paper's asynchronous one-step Sarsa)
    cuda_graphs = True                   # capture predict / observe(+update) as CUDA graphs (a3c, nstep_q, sarsa)
    max_graphs = 1024                    # cap of the graph cache; beyond it the loop runs eagerly
    DQN_type = 'nips'                    # network.py:30-55 trunk: 'nips' (agent.py:226-252) | 'nature'
    collective = 'auto'                  # gradient exchange: 'p2p' (NVLink peer memory, fused into the update) |
                                         # 'library' (arl_allreduce_grads: NCCL inside the .so) | 'torch' |
                                         # 'auto' = p2p on 2 GPUs, library beyond (measured: profiles/r02_exchange.txt)


class EnvironmentConfig(object):
    env_name = 'Breakout-v0'

    screen_width = 84
    screen_height = 84
    max_reward = 1.
    min_reward = -1.


class DQNConfig(AgentConfig, EnvironmentConfig):
    model = ''
    pass


class M1(DQNConfig):
    backend = 'b200'
    env_type = 'detail'
    action_repeat = 1


def get_config(FLAGS):
    """config.py:52-66: copy every flag whose name is a config attribute.
    FLAGS may be an argparse.Namespace, a dict, or a tf.app.flags-like object."""
    if isinstance(FLAGS, dict):
        items = dict(FLAGS)
    elif hasattr(FLAGS, '__dict__') and '__flags' in FLAGS.__dict__:
        items = dict(FLAGS.__dict__['__flags'])
    else:
        items = dict(vars(FLAGS))
    model = items.get('model', 'm1')
    if model == 'm1':
        config = type('M1', (M1,), {})   # fresh subclass: the reference mutates the class itself
    else:
        raise ValueError('unknown model: %s' % model)

    for k, v in items.items():
        if k == 'gpu':
            config.cnn_format = 'NHWC' if v is False else 'NCHW'
        if hasattr(config, k) and v is not None:
            setattr(config, k, v)
    return config
