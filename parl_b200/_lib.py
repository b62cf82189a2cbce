"""ctypes binding of libparl_b200.so — the thin shim between PyTorch-held device
memory and the C ABI declared in include/parl_b200.h.

There is NO fallback: if the library is missing or a call fails, a RuntimeError
is raised.  Tensors are passed as raw device pointers (``tensor.data_ptr()``) and
the current torch CUDA stream as ``cudaStream_t``.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'csrc', 'libparl_b200.so')

_lib = None

c_f = ctypes.c_float
c_i = ctypes.c_int
c_p = ctypes.c_void_p
c_sz = ctypes.c_size_t
c_u64 = ctypes.c_uint64
c_u32 = ctypes.c_uint32
c_i64 = ctypes.c_int64

# name -> (restype, argtypes); must list every symbol include/parl_b200.h declares
SIGNATURES = {
    'rl_abi_version': (c_i, []),
    'rl_last_error': (ctypes.c_char_p, []),
    'rl_device_sm_count': (c_i, [c_i]),
    'rl_set_sm_limit': (c_i, [c_i]),
    'rl_loss_workspace_bytes': (c_sz, [c_i]),
    'rl_debug_set_tma': (c_i, [c_i]),
    'rl_debug_set_pdl': (c_i, [c_i]),
    'rl_debug_set_vtrace_path': (c_i, [c_i]),
    'rl_vtrace_from_importance_weights': (c_i, [c_p] * 6 + [c_i, c_i, c_f, c_f, c_p, c_p, c_p]),
    'rl_vtrace_loss_fwd_bwd': (c_i, [c_p, c_p, c_p, c_i, c_p, c_p, c_p, c_i, c_i, c_i, c_i,
                                     c_f, c_f, c_f, c_f, c_f, c_p, c_p, c_p, c_p, c_p, c_p, c_sz, c_p]),
    'rl_env_atari_synth_step': (c_i, [c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i,
                                      c_i, c_i, c_u64, c_u32, c_p, c_u32, c_f, c_i, c_p]),
    'rl_env_atari_synth_step_gather': (c_i, [c_p, c_i, c_p, c_p, c_p, c_p, c_p, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p,
                                             c_i, c_i, c_u64, c_u32, c_p, c_u32, c_f, c_p, c_p]),
    'rl_obs_stack_gather': (c_i, [c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_f, c_p, c_p]),
    'rl_env_mujoco_synth_step': (c_i, [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i,
                                       c_u64, c_u32, c_u32, c_f, c_i, c_p]),
    'rl_env_cartpole_step': (c_i, [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_i,
                                   c_u64, c_u32, c_u32, c_i, c_p]),
    'rl_vecnormalize_step': (c_i, [c_p] * 12 + [c_i] * 6 + [ctypes.c_double] * 4 + [c_p]),
    'rl_sample_categorical': (c_i, [c_p, c_i, c_i, c_u64, c_u32, c_u32, c_p, c_p, c_p]),
    'rl_sample_gaussian': (c_i, [c_p, c_p, c_i, c_i, c_u64, c_u32, c_u32, c_p, c_p, c_p]),
    'rl_flat_workspace_bytes': (c_sz, [ctypes.c_longlong, c_i]),
    'rl_a2c_loss_fwd_bwd': (c_i, [c_p, c_p, c_p, c_i, c_p, c_p, ctypes.c_longlong, c_i, c_f, c_f, c_p, c_p, c_p,
                                  c_p, c_sz, c_p]),
    'rl_gae_scan_segments': (c_i, [c_p, c_p, c_p, c_p, c_i, c_i, ctypes.c_double, ctypes.c_double, c_p, c_p, c_p]),
    'rl_gae_scan': (c_i, [c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_f, c_f, c_p, c_p, c_p]),
    'rl_adv_stats': (c_i, [c_p, ctypes.c_longlong, c_p, c_p]),
    'rl_ppo_loss_fwd_bwd': (c_i, [c_p, c_p, c_p, c_p, c_i, c_p, c_p, c_p, c_p, c_p, c_p, ctypes.c_longlong, c_i,
                                  c_f, c_f, c_f, c_i, c_p, c_p, c_p, c_p, c_p, c_sz, c_p]),
    'rl_td_loss_fwd_bwd': (c_i, [c_p, c_p, c_p, c_p, c_i, c_p, c_p, c_p, ctypes.c_longlong, c_i, c_f, c_p, c_p,
                                 c_p, c_p, c_sz, c_p]),
    'rl_pg_loss_fwd_bwd': (c_i, [c_p, c_p, c_i, c_p, ctypes.c_longlong, c_i, c_p, c_p, c_p, c_sz, c_p]),
    'rl_twin_q_td_loss_fwd_bwd': (c_i, [c_p, c_p, c_p, c_p, c_p, c_p, c_p, ctypes.c_longlong, c_f, c_f, c_p, c_p, c_p, c_p,
                                        c_p, c_sz, c_p]),
    'rl_per_store': (c_i, [c_p, c_p, c_i, c_i, c_i, c_p, ctypes.c_double, ctypes.c_double, c_p]),
    'rl_per_update': (c_i, [c_p, c_p, c_i, c_p, c_p, c_i, ctypes.c_double, ctypes.c_double, c_p]),
    'rl_per_sample': (c_i, [c_p, c_p, c_i, c_i, c_p, c_u64, c_u32, ctypes.c_double, ctypes.c_double, c_p, c_p,
                            c_p, c_p]),
    'rl_replay_gather_frames': (c_i, [c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_p, c_p]),
    'rl_gather_rows': (c_i, [c_p, c_p, ctypes.c_longlong, c_i, c_p, c_p]),
    'rl_grad_global_norm': (c_i, [c_p, ctypes.c_longlong, c_p, c_p, c_sz, c_p]),
    'rl_gather_cast': (c_i, [c_p, c_p, ctypes.c_longlong, c_p, c_i, c_p]),
    'rl_adam_step': (c_i, [c_p, c_p, c_p, c_p, ctypes.c_longlong, c_p, c_f, c_f, c_f, c_f, c_i, c_f, c_p, c_f, c_i,
                           c_i, c_p, c_p]),
    'rl_gemm_bf16_tn': (c_i, [c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_i, c_i, c_p]),
    'rl_gemm_bf16_tn_splitk': (c_i, [c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_i, c_i, c_p, c_sz, c_p]),
    'rl_conv2d_nhwc_bf16_fwd': (c_i, [c_p, c_p, c_p, c_p] + [c_i] * 10 + [c_p]),
    'rl_conv2d_s1_nhwc_bf16_fwd': (c_i, [c_p, c_p, c_p, c_p] + [c_i] * 9 + [c_p]),
    'rl_conv2d_s1_u8in_bf16_fwd': (c_i, [c_p, c_f, c_p, c_p, c_p] + [c_i] * 8 + [c_p]),
    'rl_debug_set_shiftconv_base_offset': (c_i, [c_i]),
    'rl_debug_set_shiftconv_form': (c_i, [c_i]),
    'rl_debug_set_gemm_cluster': (c_i, [c_i]),
    'rl_debug_set_heads_mma': (c_i, [c_i]),
    'rl_gemm_bf16_tn_heads': (c_i, [c_p, c_p, c_p, c_p] + [c_i] * 7 + [c_p, c_p, c_i, c_p, c_i, c_p, c_sz, c_p]),
    'rl_conv2d_s1_nhwc_bf16_dgrad': (c_i, [c_p, c_p, c_p, c_p] + [c_i] * 10 + [c_p]),
    'rl_conv_wgrad_workspace_bytes': (c_sz, [c_i, c_i, c_i]),
    'rl_conv2d_s1_nhwc_bf16_wgrad': (c_i, [c_p, c_p, c_p, c_p] + [c_i] * 8 + [c_p, c_sz, c_p]),
    'rl_conv2d_s1_u8in_bf16_wgrad': (c_i, [c_p, c_p, c_f, c_p, c_p] + [c_i] * 7 + [c_p, c_sz, c_p]),
    'rl_debug_set_wgrad_lane_map': (c_i, [c_i]),
    'rl_colsum_bf16': (c_i, [c_p, ctypes.c_longlong, c_i, c_p, c_p, c_sz, c_p]),
    'rl_gemm_bf16_tn_masked': (c_i, [c_p, c_p, c_p, c_p] + [c_i] * 8 + [c_p]),
    'rl_bias_act_bf16': (c_i, [c_p, c_p, ctypes.c_longlong, c_i, c_i, c_p]),
    'rl_mlp_workspace_bytes': (c_sz, [c_i, c_p]),
    'rl_mlp_fwd': (c_i, [c_p, c_i, c_i, c_p, c_i, c_p, c_p, c_p, c_p, c_i, c_p, c_p, c_i, c_p]),
    'rl_mlp_bwd': (c_i, [c_p, c_i, c_i, c_p, c_i, c_p, c_p, c_p, c_p, c_i, c_p, c_p, c_i, c_p, c_p, c_i, c_p, c_sz, c_p]),
    'rl_rollout_mlp': (c_i, [c_i, c_p, c_i, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_i, c_p, c_p,
                             c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_u64, c_u32, c_u32, c_f, c_i, c_p, c_p, c_p, c_p, c_p,
                             c_p, c_p, c_p, c_p, c_i, c_p]),
    'rl_explore_mlp': (c_i, [c_i, c_p, c_i, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_f, c_p, c_p, c_p, c_p,
                             c_p, c_p, c_p, c_i, c_u64, c_u32, c_u32, c_f, c_i, c_p, c_p, c_p, c_p, c_p, c_i, c_i,
                             c_p]),
    'rl_replay_sample_uniform': (c_i, [c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_p, c_p, c_i, c_i, c_u64, c_p, c_p, c_p, c_p,
                                       c_p, c_p, c_p]),
    'rl_mask_scatter_grid_bf16': (c_i, [c_p, c_p, c_p, ctypes.c_longlong, c_i, c_i, c_i, c_i, c_i, c_p]),
}


def load():
    """Load the shared library (building is a separate, explicit step)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            'parl_b200: CUDA library %s not found. Build it with `python -m parl_b200.build` '
            '(there is no CPU fallback).' % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    # triage switches from the environment (defaults live in the library)
    if os.environ.get('PARL_B200_PDL', '') == '1':
        lib.rl_debug_set_pdl(1)
    if os.environ.get('PARL_B200_GEMM_CLUSTER', '') == '0':
        lib.rl_debug_set_gemm_cluster(0)
    if os.environ.get('PARL_B200_HEADS_MMA', '') == '0':
        lib.rl_debug_set_heads_mma(0)
    return lib


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    return ctypes.c_void_p(t.data_ptr())


def stream():
    """cudaStream_t of torch's current stream on the current device.  Launches are made on the current device:
    ``require_cuda`` rejects tensors that live on another GPU (one process drives one GPU, SURVEY.md 8e)."""
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


launches = 0          # number of C-ABI kernel-launching calls made by this process (bench.py gpu_launches)


def check(code, what):
    global launches
    launches += 1
    if code != 0:
        msg = load().rl_last_error().decode()
        raise RuntimeError('parl_b200.%s failed (code %d): %s' % (what, code, msg))


def check_config(code, what):
    """check() for calls that only set a library switch (no kernel launch: not counted in ``launches``)."""
    global launches
    check(code, what)
    launches -= 1


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError('parl_b200 kernels need CUDA tensors (no CPU fallback); got a %s tensor' % t.device)
        if t is not None and not t.is_contiguous():
            raise RuntimeError('parl_b200 kernels need contiguous tensors')
        if t is not None and t.device.index != torch.cuda.current_device():
            # launches go to the current device's current stream; a tensor of another GPU would be dereferenced
            # from the wrong context (ADVICE r1): make the owner set the device (torch.cuda.set_device / device guard)
            raise RuntimeError('parl_b200: tensor on cuda:%d but the current device is cuda:%d — wrap the call in '
                               'torch.cuda.device(tensor.device)' % (t.device.index, torch.cuda.current_device()))
