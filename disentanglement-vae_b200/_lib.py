"""ctypes binding of the C ABI declared in `include/dvae_b200.h`.

The library is built in-tree (`__graft_entry__.build()` -> `disentanglement-vae_b200/libdvae_b200.so`).
There is NO fallback: if the library is missing or a call fails, a `DvaeError` is raised.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdvae_b200.so")

MAX_SPACES = 8
HEADS_NSCALARS = 3 + 3 * MAX_SPACES


class DvaeError(RuntimeError):
    pass


_p = C.c_void_p
_i = C.c_int
_l = C.c_int64
_f = C.c_float
_u32 = C.c_uint32
_pp = C.POINTER(C.c_void_p)
_ip = C.POINTER(C.c_int)

# name -> (restype, argtypes); mirrors include/dvae_b200.h one-to-one
SIGNATURES = {
    "dvae_last_error_string": (C.c_char_p, []),
    "dvae_version": (_i, []),
    "dvae_launch_count": (_l, []),
    "dvae_weight_planes_floats": (_l, [_i, _i, _i]),
    "dvae_weight_planes_register": (_i, [_p, _i, _i, _p, _p]),
    "dvae_weight_planes_refresh": (_i, [_p]),
    "dvae_weight_planes_refresh_ex": (_i, [_i, _i, _p]),
    "dvae_weight_planes_enable": (_i, [_i]),
    "dvae_weight_planes_clear": (_i, []),
    "dvae_defer_joins": (_i, [_i]),
    "dvae_join_side_streams": (_i, [_p]),
    "dvae_linear": (_i, [_p, _l, _i, _p, _l, _i, _p, _l, _i, _i, _i, _p, _p, _f, _i, _p]),
    "dvae_tc_linear": (_i, [_p, _l, _i, _p, _l, _i, _p, _l, _i, _i, _i, _p, _p, _f, _i, _i, _p]),
    "dvae_tc16_linear": (_i, [_p, _l, _i, _p, _l, _i, _p, _l, _i, _i, _i, _p, _p, _f, _i, _f, _f, _p, _p, _p]),
    "dvae_colsum": (_i, [_p, _l, _i, _i, _p, _f, _p]),
    "dvae_randn": (_i, [_p, _l, _p, _u32, _p]),
    "dvae_embedding_fwd": (_i, [_p, _i, _p, _l, _l, _i, _i, _f, _p, _u32, _l, _i, _p, _p]),
    "dvae_embedding_bwd": (_i, [_p, _i, _p, _l, _l, _i, _i, _f, _p, _u32, _l, _i, _p, _p]),
    "dvae_bow_encoder_fwd": (_i, [_p, _i, _p, _l, _l, _i, _i, _f, _p, _u32, _p, _l, _p, _p]),
    "dvae_bow_encoder_bwd": (_i, [_p, _l, _p, _i, _p, _l, _l, _i, _i, _f, _p, _u32, _p, _p]),
    "dvae_dropout": (_i, [_p, _l, _l, _i, _f, _p, _u32, _p, _l, _l, _p]),
    "dvae_lstm_step": (_i, [_p, _l, _i, _i, _i, _i, _i, _p, _p, _p, _p, _p, _p, _l, _p, _p, _p, _p, _p]),
    "dvae_vocab_sample_step": (_i, [_p, _l, _i, _i, _i, _p, _p, _p, _u32, _p, _l, _p, _p]),
    "dvae_vocab_sample_step_ex": (_i, [_p, _l, _i, _i, _i, _p, _p, _p, _u32, _p, _l, _p, _p, _p]),
    "dvae_vocab_w_planes_floats": (_l, [_i, _i]),
    "dvae_vocab_w_planes": (_i, [_p, _i, _i, _p, _p]),
    "dvae_vocab_sample_step_planes": (_i, [_p, _l, _i, _i, _i, _p, _p, _p, _p, _u32, _p, _l, _p, _p, _p]),
    "dvae_recount_lengths": (_i, [_p, _l, _l, _i, _i, _l, _l, _l, _p, _p]),
    "dvae_bleu_counts": (_i, [_p, _l, _i, _p, _l, _i, _i, _l, _p, _p]),
    "dvae_bleu_score": (_i, [_p, _p, _p]),
    "dvae_lstm_state_ws_floats": (_l, [_i, _i, _i]),
    "dvae_lstm_seq_fwd": (_i, [_p, _l, _i, _i, _i, _i, _i, _pp, _pp, _pp, _pp, _p, _p, _l, _l, _p, _p, _l, _p, _p,
                               _l, _l, _p, _p, _p, _p]),
    "dvae_lstm_input_proj": (_i, [_p, _l, _i, _i, _i, _i, _i, _pp, _pp, _pp, _p, _p]),
    "dvae_lstm_seq_fwd_ex": (_i, [_p, _l, _i, _i, _i, _i, _i, _pp, _pp, _pp, _pp, _p, _p, _l, _l, _p, _p, _l, _p, _p,
                                  _l, _l, _p, _p, _p, _i, _p]),
    "dvae_lstm_seq_bwd": (_i, [_p, _l, _i, _i, _i, _i, _i, _pp, _pp, _p, _p, _l, _l, _p, _p, _l, _p, _p, _p, _l,
                               _p, _p, _l, _l, _p, _l, _pp, _pp, _pp, _pp, _p, _p, _l, _l, _p, _p]),
    "dvae_lstm_bwd_planes_ws_floats": (_l, [_i, _i, _i, _i, _i]),
    "dvae_lstm_seq_bwd_ex": (_i, [_p, _l, _i, _i, _i, _i, _i, _pp, _pp, _p, _p, _l, _l, _p, _p, _l, _p, _p, _p, _l,
                                  _p, _p, _l, _l, _p, _l, _pp, _pp, _pp, _pp, _p, _p, _l, _l, _p, _p, _p]),
    "dvae_counter_increment": (_i, [_p, _p]),
    "dvae_fork_after": (_i, [_i, _p, _p, C.POINTER(C.c_void_p)]),
    "dvae_nvls_barrier_words": (_l, []),
    "dvae_nvls_all_reduce": (_i, [_p, _l, _pp, _i, _i, _p, C.c_uint32, C.c_uint32, _i, C.c_uint64, _p, _p]),
    "dvae_p2p_all_reduce": (_i, [_pp, _l, _pp, _i, _i, _p, C.c_uint32, C.c_uint32, _i, C.c_uint64, _p, _p]),
    "dvae_heads_ws_floats": (_l, [_i, _i]),
    "dvae_latent_heads_fwd": (_i, [_p, _i, _i, _i, _ip, _ip, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i, _p, _p, _p,
                                   _p, _p, _p, _p, _p]),
    "dvae_heads_bwd_ws_floats": (_l, [_i, _i, _i]),
    "dvae_latent_heads_bwd": (_i, [_p, _i, _i, _i, _ip, _ip, _p, _p, _p, _p, _p, _p, _i, _p, _p, _p, _p, _p, _p,
                                   _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "dvae_dsc_loss": (_i, [_p, _p, _i, _i, _ip, _ip, _p, _p, _p, _p]),
    "dvae_vocab_ce_ws_floats": (_l, [_i, _i, _i]),
    "dvae_vocab_ce_fwd": (_i, [_p, _l, _i, _i, _i, _i, _p, _p, _p, _l, _p, _i, _p, _p, _p, _p, _p, _p]),
    "dvae_vocab_split_w": (_i, [_p, _i, _i, _i, _p, _p]),
    "dvae_vocab_ce_fwd_ex": (_i, [_p, _l, _i, _i, _i, _i, _p, _p, _p, _l, _p, _i, _p, _p, _p, _p, _p, _i, _p]),
    "dvae_vocab_ce_partials": (_i, [_p, _l, _i, _i, _i, _i, _p, _p, _p, _l, _p, _i, _p, _p]),
    "dvae_vocab_ce_fwd_live": (_i, [_p, _l, _i, _i, _i, _i, _p, _p, _p, _l, _p, _i, _p, _p, _p, _p, _p, _i, _p]),
    "dvae_vocab_live_rows_at": (_l, [_i, _i, _i]),
    "dvae_vocab_ce_bwd_ws_floats": (_l, [_i, _i, _i]),
    "dvae_vocab_ce_bwd": (_i, [_p, _l, _i, _i, _i, _i, _p, _p, _p, _l, _p, _p, _p, _p, _l, _p, _p, _p, _p, _p]),
    "dvae_vocab_ce_bwd_live": (_i, [_p, _l, _i, _i, _i, _i, _p, _p, _p, _l, _p, _p, _p, _p, _l, _p, _p, _p, _p, _p]),
    "dvae_entropy_loss": (_i, [_p, _i, _i, _p, _p, _p, _p]),
    "dvae_club_mi": (_i, [_p, _p, _p, _i, _i, _p, _p, _p, _p, _p, _p, _p]),
    "dvae_club_nll": (_i, [_p, _p, _p, _i, _i, _p, _p, _p, _p, _p]),
    "dvae_act_bwd": (_i, [_p, _p, _p, _l, _i, _p]),
    "dvae_relu": (_i, [_p, _l, _p]),
    "dvae_grad_sumsq": (_i, [_p, _l, _p, _p, _p]),
    "dvae_clip_adam": (_i, [_p, _p, _p, _p, _l, _p, _f, _f, _p, _i, _p]),
}

_lib = None
planes_owner = None      # id() of the engine whose weights are in the library's weight-plane registry (engine.py)


def load():
    """Load (once) and return the ctypes handle; raises DvaeError if the extension is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DvaeError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  There is no CPU or PyTorch fallback for this path.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise DvaeError(f"{LIB_PATH} does not export {name}") from e
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().dvae_last_error_string()
        raise DvaeError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def ptr_array(tensors):
    """Host array of device pointers (const float* const*)."""
    arr = (C.c_void_p * max(len(tensors), 1))()
    for i, t in enumerate(tensors):
        arr[i] = None if t is None else t.data_ptr()
    return arr


def int_array(vals):
    arr = (C.c_int * max(len(vals), 1))()
    for i, v in enumerate(vals):
        arr[i] = int(v)
    return arr


def stream_ptr():
    import torch
    return torch.cuda.current_stream().cuda_stream


def launch_count():
    return int(load().dvae_launch_count())
