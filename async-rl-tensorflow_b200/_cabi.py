"""ctypes binding of libasyncrl_b200.so (include/asyncrl_b200.h, include/asyncrl_b200_sarsa.h,
include/asyncrl_b200_dueling.h, include/asyncrl_b200_double.h, include/asyncrl_b200_dueling_streams.h,
include/asyncrl_b200_lstm.h).

The product path has no CPU fallback: if the shared library is missing or a call
fails, this module raises.  PyTorch is only the carrier of device memory and
streams; every tensor is handed to the library as a raw device pointer.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libasyncrl_b200.so")

c_int, c_i64, c_u64, c_f32, c_vp = (ctypes.c_int, ctypes.c_int64, ctypes.c_uint64,
                                     ctypes.c_float, ctypes.c_void_p)

# name -> argtypes (all return int except where noted); mirrors include/asyncrl_b200.h
SIGNATURES = {
    "arl_init": [c_int],
    "arl_param_layout": [c_int, ctypes.POINTER(c_i64)],
    "arl_preprocess_push": [c_vp, c_vp, c_int, c_int, c_int, c_int, c_vp],
    "arl_preprocess_push_pil": [c_vp, c_vp, c_int, c_int, c_int, c_int, c_vp],
    "arl_upload_frames": [c_vp, c_vp, c_int, c_vp],
    "arl_upload_frames_full": [c_vp, c_vp, c_int, c_vp],
    "arl_history_get": [c_vp, c_vp, c_int, c_int, c_int, c_int, c_vp],
    "arl_history_reset": [c_vp, c_int, c_int, c_vp],
    "arl_conv1_forward": [c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_vp],
    "arl_conv2_forward": [c_vp, c_vp, c_vp, c_i64, c_vp],
    "arl_prepare_weights": [c_vp, c_vp, c_vp],
    "arl_fc_forward": [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp],
    "arl_heads_forward": [c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp],
    "arl_forward": [c_vp, c_vp, c_int, c_int, c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp,
                    c_vp, c_vp, c_vp, c_vp],
    "arl_fc_heads_forward": [c_vp, c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_u64,
                             c_i64, c_vp],
    "arl_forward_sample": [c_vp, c_vp, c_int, c_int, c_vp, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp,
                           c_vp, c_vp, c_i64, c_i64, c_vp, c_u64, c_vp],
    "arl_forward_egreedy": [c_vp, c_vp, c_int, c_int, c_vp, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp,
                            c_vp, c_vp, c_i64, c_i64, c_vp, c_u64, c_f32, ctypes.c_double, ctypes.c_double,
                            ctypes.c_double, ctypes.c_double, c_vp],
    "arl_debug_gemm": [c_int, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_vp],
    "arl_sample_actions": [c_vp, c_vp, c_int, c_int, c_i64, c_i64, c_u64, c_vp],
    "arl_greedy_actions": [c_vp, c_vp, c_int, c_int, c_vp],
    "arl_egreedy_actions": [c_vp, c_vp, c_int, c_int, c_f32, c_i64, c_i64, c_u64, c_vp],
    "arl_act_update": [c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_vp, c_int, c_vp],
    "arl_observe_store": [c_vp, c_vp, c_vp, c_vp, c_int, c_vp],
    "arl_q_lossgrad": [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_f32, c_f32,
                       c_f32, c_f32, c_vp],
    "arl_nstep_q_lossgrad": [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_f32, c_f32,
                             c_f32, c_f32, c_vp],
    "arl_returns_lossgrad": [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int,
                             c_int, c_int, c_f32, c_f32, c_f32, c_f32, c_f32, c_vp],
    "arl_heads_backward": [c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_f32, c_vp],
    "arl_fc_backward": [c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_i64, c_f32, c_vp],
    "arl_conv2_backward": [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_f32, c_vp],
    "arl_conv1_backward": [c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_f32, c_vp],
    "arl_backward": [c_vp, c_vp, c_int, c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp,
                     c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_f32, c_int, c_vp],
    "arl_sample_actions_dev": [c_vp, c_vp, c_int, c_int, c_i64, c_vp, c_u64, c_vp],
    "arl_step_advance": [c_vp, c_i64, c_vp],
    "arl_observe_store_advance": [c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_i64, c_vp],
    "arl_clip_rmsprop_sched": [c_vp, c_vp, c_vp, c_int, c_vp, c_i64, ctypes.c_double, c_i64, c_f32, c_f32,
                               c_f32, c_vp, c_vp, c_vp],
    "arl_nature_param_layout": [c_int, ctypes.POINTER(c_i64)],
    "arl_nature_forward": [c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp],
    "arl_nature_backward": [c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                            c_vp, c_vp, c_i64, c_vp],
    "arl_clip_rmsprop_layout": [c_vp, c_vp, c_vp, ctypes.POINTER(c_i64), c_int, c_f32, c_vp, c_i64,
                                ctypes.c_double, c_i64, c_f32, c_f32, c_f32, c_vp, c_vp, c_vp],
    "arl_comm_enable_p2p": [c_i64],
    "arl_exchange_clip_rmsprop": [c_vp, c_vp, c_vp, ctypes.POINTER(c_i64), c_int, c_f32, c_vp, c_i64,
                                  ctypes.c_double, c_i64, c_f32, c_f32, c_f32, c_vp, c_vp, c_vp],
    "arl_comm_unique_id": [c_vp],
    "arl_comm_init": [c_vp, c_int, c_int],
    "arl_comm_destroy": [],
    "arl_allreduce_grads": [c_vp, c_i64, c_vp],
    "arl_allreduce_begin": [c_vp, c_i64, c_i64, c_vp],
    "arl_allreduce_end": [c_vp],
    "arl_clip_rmsprop": [c_vp, c_vp, c_vp, c_int, c_f32, c_f32, c_f32, c_f32, c_vp, c_vp, c_vp],
}
OTHER = {
    "arl_last_error": ([], ctypes.c_char_p),
    "arl_version": ([], c_int),
    "arl_backward_workspace_bytes": ([c_int], c_i64),
    "arl_prepared_floats": ([], c_i64),
    "arl_a2_block_rows": ([c_int], c_i64),
    "arl_launch_count": ([c_int], c_i64),
    "arl_nature_workspace_bytes": ([c_int], c_i64),
    "arl_comm_size": ([], c_int),
    "arl_comm_p2p_enabled": ([], c_int),
    "arl_comm_p2p_error": ([], c_int),
    "arl_comm_nccl_version": ([], c_int),
}
EXPORTS = tuple(SIGNATURES) + tuple(OTHER)

# the one-step Sarsa entry: its own header (include/asyncrl_b200_sarsa.h), its own table
SARSA_SIGNATURES = {
    "arl_sarsa_lossgrad": [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_f32, c_f32,
                           c_f32, c_f32, c_vp],
}

# the dueling Q heads: their own header (include/asyncrl_b200_dueling.h), their own table
DUELING_SIGNATURES = {
    "arl_forward_dueling": [c_vp, c_vp, c_int, c_int, c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp,
                            c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_u64, c_f32, ctypes.c_double, ctypes.c_double,
                            ctypes.c_double, ctypes.c_double, c_vp],
    "arl_q_lossgrad_dueling": [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_f32, c_f32,
                               c_f32, c_f32, c_vp],
    "arl_nstep_q_lossgrad_dueling": [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int,
                                     c_f32, c_f32, c_f32, c_f32, c_vp],
    "arl_sarsa_lossgrad_dueling": [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int,
                                   c_f32, c_f32, c_f32, c_f32, c_vp],
}

# the double Q-learning targets: their own header (include/asyncrl_b200_double.h), their own table
DOUBLE_SIGNATURES = {
    "arl_double_q_lossgrad": [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_f32,
                              c_f32, c_f32, c_f32, c_vp],
    "arl_double_q_lossgrad_dueling": [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int,
                                      c_int, c_f32, c_f32, c_f32, c_f32, c_vp],
    "arl_double_nstep_q_lossgrad": [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int,
                                    c_f32, c_f32, c_f32, c_f32, c_vp],
    "arl_double_nstep_q_lossgrad_dueling": [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int,
                                            c_int, c_int, c_f32, c_f32, c_f32, c_f32, c_vp],
}

# the dueling streams (a hidden layer per stream): their own header (include/asyncrl_b200_dueling_streams.h),
# their own tables
STREAMS_SIGNATURES = {
    "arl_streams_param_layout": [c_int, ctypes.POINTER(c_i64)],
    "arl_prepare_weights_streams": [c_vp, c_vp, c_int, c_vp],
    "arl_fc_forward_streams": [c_vp, c_vp, c_vp, c_i64, c_vp],
    "arl_forward_streams": [c_vp, c_vp, c_int, c_int, c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp,
                            c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_u64, c_f32, ctypes.c_double, ctypes.c_double,
                            ctypes.c_double, ctypes.c_double, c_vp],
    "arl_heads_backward_streams": [c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_f32, c_vp],
    "arl_fc_backward_streams": [c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_i64, c_f32, c_int, c_vp],
    "arl_backward_streams": [c_vp, c_vp, c_int, c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                             c_vp, c_vp, c_vp, c_vp, c_f32, c_int, c_vp],
}
STREAMS_OTHER = {
    "arl_streams_prepared_floats": ([], c_i64),
    "arl_streams_workspace_bytes": ([c_int], c_i64),
}

# the A3C LSTM agent: its own header (include/asyncrl_b200_lstm.h), its own tables
LSTM_SIGNATURES = {
    "arl_lstm_param_layout": [c_int, ctypes.POINTER(c_i64)],
    "arl_prepare_weights_lstm": [c_vp, c_vp, c_int, c_vp],
    "arl_lstm_step": [c_vp, c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int,
                      c_vp],
    "arl_forward_lstm": [c_vp, c_vp, c_int, c_int, c_vp, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                         c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_u64,
                         c_vp],
    "arl_heads_backward_lstm": [c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_f32, c_vp],
    "arl_lstm_backward": [c_vp, c_vp, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                          c_vp, c_vp, c_vp, c_vp, c_f32, c_vp],
    "arl_backward_lstm": [c_vp, c_vp, c_int, c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                          c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_f32,
                          c_int, c_vp],
}
LSTM_OTHER = {
    "arl_lstm_prepared_floats": ([], c_i64),
    "arl_lstm_workspace_bytes": ([c_int], c_i64),
}


class ArlError(RuntimeError):
    pass


_lib = None
_inited = set()


def load():
    """dlopen the in-tree library (no GPU needed) and declare the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ArlError("%s is missing: build it with async-rl-tensorflow_b200/csrc/build.sh "
                       "(or __graft_entry__.build()); there is no CPU fallback" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, argtypes in (list(SIGNATURES.items()) + list(SARSA_SIGNATURES.items())
                           + list(DUELING_SIGNATURES.items()) + list(DOUBLE_SIGNATURES.items())
                           + list(STREAMS_SIGNATURES.items()) + list(LSTM_SIGNATURES.items())):
        fn = getattr(lib, name)
        fn.argtypes, fn.restype = argtypes, c_int
    for name, (argtypes, restype) in list(OTHER.items()) + list(STREAMS_OTHER.items()) + list(LSTM_OTHER.items()):
        fn = getattr(lib, name)
        fn.argtypes, fn.restype = argtypes, restype
    _lib = lib
    return lib


def check(rc, name):
    if rc != 0:
        raise ArlError("%s failed (%d): %s" % (name, rc, load().arl_last_error().decode()))


def init(device):
    """arl_init once per device.  Raises if there is no CUDA device."""
    if not torch.cuda.is_available():
        raise ArlError("asyncrl_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    idx = torch.device(device).index
    if idx is None:
        idx = torch.cuda.current_device()
    if idx not in _inited:
        check(load().arl_init(idx), "arl_init")
        _inited.add(idx)
    return idx


def ptr(t):
    """Raw device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise ArlError("expected a CUDA tensor, got device %s" % t.device)
    if not t.is_contiguous():
        raise ArlError("expected a contiguous tensor")
    return t.data_ptr()


def stream_ptr():
    return torch.cuda.current_stream().cuda_stream


def call(name, *args):
    check(getattr(load(), name)(*args), name)


def param_layout(action_size):
    """(names, offsets[11]) of the flat parameter buffer."""
    off = (c_i64 * 11)()
    check(load().arl_param_layout(int(action_size), off), "arl_param_layout")
    return list(off)


def nature_param_layout(action_size):
    """Offsets (13) of the 'nature' flat parameter buffer."""
    off = (c_i64 * 13)()
    check(load().arl_nature_param_layout(int(action_size), off), "arl_nature_param_layout")
    return list(off)


def streams_param_layout(action_size):
    """Offsets (13) of the dueling streams' flat parameter buffer: arl_param_layout's 10 tensors, then la_w,
    la_b."""
    off = (c_i64 * 13)()
    check(load().arl_streams_param_layout(int(action_size), off), "arl_streams_param_layout")
    return list(off)


def lstm_param_layout(action_size):
    """Offsets (13) of the LSTM network's flat parameter buffer: arl_param_layout's 10 tensors, then lstm_w,
    lstm_b."""
    off = (c_i64 * 13)()
    check(load().arl_lstm_param_layout(int(action_size), off), "arl_lstm_param_layout")
    return list(off)


def a2_block_rows(num_envs):
    """Rows of one a2 block (envs per forward launch): see arl_a2_block_rows."""
    return int(load().arl_a2_block_rows(int(num_envs)))


def launch_count(reset=False):
    """Kernels launched by the library so far in this process."""
    return int(load().arl_launch_count(1 if reset else 0))


def prepared_floats(streams=False, lstm=False):
    """Size (floats) of the prepared-weights buffer arl_prepare_weights (``streams``:
    arl_prepare_weights_streams, ``lstm``: arl_prepare_weights_lstm) fills."""
    if lstm:
        return int(load().arl_lstm_prepared_floats())
    if streams:
        return int(load().arl_streams_prepared_floats())
    return int(load().arl_prepared_floats())


def workspace_bytes(action_size, streams=False, lstm=False):
    if lstm:
        return int(load().arl_lstm_workspace_bytes(int(action_size)))
    if streams:
        return int(load().arl_streams_workspace_bytes(int(action_size)))
    return int(load().arl_backward_workspace_bytes(int(action_size)))


def comm_size():
    """Ranks of the library's communicator (0 = arl_comm_init has not been called)."""
    return int(load().arl_comm_size())


def comm_init(device):
    """arl_comm_init for this process from the torch.distributed world: rank 0 makes the NCCL id
    (arl_comm_unique_id), torch.distributed carries its 128 bytes to the other ranks -- plumbing
    only; the gradients themselves never go through torch."""
    import torch.distributed as dist
    if comm_size():
        return comm_size()
    rank, world = dist.get_rank(), dist.get_world_size()
    buf = ctypes.create_string_buffer(128)
    if rank == 0:
        check(load().arl_comm_unique_id(buf), "arl_comm_unique_id")
    t = torch.frombuffer(bytearray(buf.raw), dtype=torch.uint8).clone()
    on_dev = dist.get_backend() == "nccl"
    if on_dev:
        t = t.to(device)
    dist.broadcast(t, 0)
    idb = ctypes.create_string_buffer(bytes(t.cpu().numpy().tobytes()), 128)
    with torch.cuda.device(device):
        check(load().arl_comm_init(idb, rank, world), "arl_comm_init")
    return world
