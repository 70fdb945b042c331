"""ctypes binding of libmelgan_b200.so (the C ABI in include/melgan_b200.h).

PyTorch is plumbing here: it owns device memory and streams; every kernel that runs on the hot
path lives in the shared library.  There is no CPU or eager-PyTorch fallback: if the library
is missing, or the device is not sm_100, calls raise.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libmelgan_b200.so")
NUM_LAYERS = 30

_f32p = ctypes.POINTER(ctypes.c_float)
_lib = None


class EngineError(RuntimeError):
    pass


def lib():
    """Loads the shared library (once).  Raises if it has not been built: the product path never
    degrades to a fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise EngineError(
                "libmelgan_b200.so is not built (%s). Run `python -m melgan_multi_b200.build` "
                "(needs nvcc); there is no CPU/PyTorch fallback for the hot path." % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        L.mg_abi_version.restype = ctypes.c_int
        L.mg_last_error_string.restype = ctypes.c_char_p
        L.mg_device_check.restype = ctypes.c_int
        L.mg_gen_packed_bytes.restype = ctypes.c_size_t
        L.mg_gen_pack.restype = ctypes.c_int
        L.mg_gen_pack.argtypes = [ctypes.c_void_p] * 5
        L.mg_gen_workspace_bytes.restype = ctypes.c_size_t
        L.mg_gen_workspace_bytes.argtypes = [ctypes.c_int, ctypes.c_int]
        L.mg_gen_forward.restype = ctypes.c_int
        L.mg_gen_forward.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                                     ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
        L.mg_gen_forward_varlen.restype = ctypes.c_int
        L.mg_gen_forward_varlen.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
                                            ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
        L.mg_gen_forward_timed.restype = ctypes.c_int
        L.mg_gen_forward_timed.argtypes = L.mg_gen_forward.argtypes + [ctypes.POINTER(ctypes.c_float)]
        L.mg_gen_check_status.restype = ctypes.c_int
        L.mg_gen_check_status.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
        L.mg_gen_convt.restype = ctypes.c_int
        L.mg_gen_convt.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                                   ctypes.c_int, ctypes.c_void_p]
        L.mg_gen_resblock.restype = ctypes.c_int
        L.mg_gen_resblock.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                                      ctypes.c_int, ctypes.c_void_p]
        L.mg_gen_upres.restype = ctypes.c_int
        L.mg_gen_upres.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                                   ctypes.c_int, ctypes.c_void_p]
        L.mg_gen_conv_pre.restype = ctypes.c_int
        L.mg_gen_conv_pre.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
        L.mg_gen_resblock_post.restype = ctypes.c_int
        L.mg_gen_resblock_post.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
        L.mg_disc_packed_bytes.restype = ctypes.c_size_t
        L.mg_disc_pack.restype = ctypes.c_int
        L.mg_disc_pack.argtypes = [ctypes.c_void_p] * 5
        L.mg_disc_forward.restype = ctypes.c_int
        L.mg_disc_forward.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                                      ctypes.c_void_p, ctypes.c_void_p]
        L.mg_gen_resup.restype = ctypes.c_int
        L.mg_gen_resup.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
                                   ctypes.c_void_p]
        L.mg_gen_set_pipeline.restype = ctypes.c_int
        L.mg_gen_set_pipeline.argtypes = [ctypes.c_int]
        L.mg_gen_stage_output.restype = ctypes.c_int
        L.mg_gen_stage_output.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int,
                                          ctypes.c_int, ctypes.c_void_p]
        L.mg_gen_forward_launches.restype = ctypes.c_int
        L.mg_gen_forward_slices.restype = ctypes.c_int
        L.mg_gen_forward_slices.argtypes = [ctypes.c_int, ctypes.c_int]
        L.mg_gen_kernel_name.restype = ctypes.c_char_p
        L.mg_gen_kernel_name.argtypes = [ctypes.c_int]
        L.mg_msd_packed_bytes.restype = ctypes.c_size_t
        L.mg_msd_pack.restype = ctypes.c_int
        L.mg_msd_pack.argtypes = [ctypes.c_void_p] * 5
        L.mg_msd_lengths.restype = ctypes.c_int
        L.mg_msd_lengths.argtypes = [ctypes.c_int, ctypes.POINTER(ctypes.c_int)]
        L.mg_msd_forward.restype = ctypes.c_int
        L.mg_msd_forward.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                                     ctypes.c_void_p, ctypes.c_void_p]
        L.mg_msd_grouped_backward_workspace_bytes.restype = ctypes.c_size_t
        L.mg_msd_grouped_backward_workspace_bytes.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int]
        L.mg_msd_grouped_backward.restype = ctypes.c_int
        L.mg_msd_grouped_backward.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int] + [ctypes.c_void_p] * 6 + [
            ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
        L.mg_msd_post1_dgrad.restype = ctypes.c_int
        L.mg_msd_post1_dgrad.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
                                         ctypes.c_void_p, ctypes.c_void_p]
        L.mg_msd_post1_wgrad.restype = ctypes.c_int
        L.mg_msd_post1_wgrad.argtypes = [ctypes.c_void_p] * 4 + [ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
        L.mg_msd_edge_backward_workspace_bytes.restype = ctypes.c_size_t
        L.mg_msd_edge_backward_workspace_bytes.argtypes = [ctypes.c_int] * 3
        L.mg_msd_edge_backward.restype = ctypes.c_int
        L.mg_msd_edge_backward.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int] + [ctypes.c_void_p] * 6 + [
            ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
        L.mg_msd_scale_backward_workspace_bytes.restype = ctypes.c_size_t
        L.mg_msd_scale_backward_workspace_bytes.argtypes = [ctypes.c_int, ctypes.c_int]
        L.mg_msd_scale_backward.restype = ctypes.c_int
        L.mg_msd_scale_backward.argtypes = [ctypes.c_void_p, ctypes.c_int] + [ctypes.c_void_p] * 8 + [
            ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
        L.mg_lrelu_backward.restype = ctypes.c_int
        L.mg_lrelu_backward.argtypes = [ctypes.c_void_p] * 4 + [ctypes.c_longlong, ctypes.c_void_p]
        L.mg_msd_wn_backward.restype = ctypes.c_int
        L.mg_msd_wn_backward.argtypes = [ctypes.c_void_p] * 6
        L.mg_adam_chunk.restype = ctypes.c_int
        L.mg_adam_step.restype = ctypes.c_int
        L.mg_adam_step.argtypes = [ctypes.c_void_p] * 6 + [ctypes.c_int, ctypes.c_int] + [ctypes.c_float] * 5 + [
            ctypes.c_longlong, ctypes.c_void_p]
        L.mg_loss_workspace_bytes.restype = ctypes.c_size_t
        L.mg_loss_workspace_bytes.argtypes = [ctypes.c_void_p, ctypes.c_int]
        L.mg_loss_forward.restype = ctypes.c_int
        L.mg_loss_forward.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                                      ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
        L.mg_loss_backward.restype = ctypes.c_int
        L.mg_loss_backward.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                                       ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        L.mg_msd_check_status.restype = ctypes.c_int
        L.mg_msd_check_status.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        L.mg_gen_engine_create.restype = ctypes.c_int
        L.mg_gen_engine_create.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.c_int, ctypes.c_int]
        L.mg_gen_engine_load_state.restype = ctypes.c_int
        L.mg_gen_engine_load_state.argtypes = [ctypes.c_void_p] * 4
        L.mg_gen_engine_forward.restype = ctypes.c_int
        L.mg_gen_engine_forward.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                                            ctypes.c_int]
        L.mg_gen_engine_forward_varlen.restype = ctypes.c_int
        L.mg_gen_engine_forward_varlen.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                                                   ctypes.c_int, ctypes.c_void_p]
        L.mg_gen_engine_last_kernel_ms.restype = ctypes.c_int
        L.mg_gen_engine_last_kernel_ms.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_float)]
        L.mg_gen_engine_destroy.restype = None
        L.mg_gen_engine_destroy.argtypes = [ctypes.c_void_p]
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise EngineError("melgan_b200 error %d: %s" % (rc, lib().mg_last_error_string().decode()))


def _ptr_array(ptrs):
    return (ctypes.c_void_p * len(ptrs))(*ptrs)


def lengths_array(lengths, B):
    """Per-item mel lengths (list, tuple, numpy array or integer torch tensor; a CUDA tensor is copied to the host, which
    synchronises with its stream) as the host int32 array the ragged entry points take.  Range checks are the library's."""
    if hasattr(lengths, "detach"):  # torch tensor
        if lengths.is_floating_point() or lengths.is_complex():
            raise EngineError("lengths must be integers, got %s" % (lengths.dtype,))
        lengths = lengths.detach().cpu().numpy()
    a = np.asarray(lengths)
    if a.ndim != 1 or a.shape[0] != B:
        raise EngineError("lengths must hold one value per batch item (%d), got shape %s" % (B, a.shape))
    if a.size and not np.issubdtype(a.dtype, np.integer):
        raise EngineError("lengths must be integers, got %s" % (a.dtype,))
    if a.size and (a.min() < np.iinfo(np.int32).min or a.max() > np.iinfo(np.int32).max):
        raise EngineError("lengths out of the int32 range")
    return (ctypes.c_int * B)(*a.astype(np.int64).tolist())


class _StatusWatch:
    """The tcgen05 kernels bound every mbarrier wait and, on a timeout, raise a device status word and carry on (a hung
    GPU box is worse than a failed call).  A forward must therefore never be trusted silently: after each one the status
    word is copied to pinned host memory on the same stream (4 bytes, asynchronous), and the copy is inspected at the
    next forward of the same module, or at the next host synchronisation point the training loop has anyway
    (``discriminator_loss``' read-back, ``poll_status``).  A non-zero word raises EngineError.  Skipped while the stream
    is being captured into a CUDA graph (no host-visible copy can be made there; replays are checked by check_status)."""
    _live = None  # weak set of watches with a copy in flight

    def __init__(self, torch, device, what):
        import weakref
        self.torch, self.what = torch, what
        self.pin = torch.zeros(1, dtype=torch.int32).pin_memory()
        self.event = torch.cuda.Event()
        self.pending = False
        if _StatusWatch._live is None:
            _StatusWatch._live = weakref.WeakSet()

    def arm(self, status_word):
        """status_word: int32 CUDA tensor view [1] holding the pipeline's status after the work just enqueued."""
        if self.torch.cuda.is_current_stream_capturing():
            return
        self.pin.copy_(status_word, non_blocking=True)
        self.event.record()
        self.pending = True
        _StatusWatch._live.add(self)

    def check(self, wait=False):
        if not self.pending or self.torch.cuda.is_current_stream_capturing():
            return  # (event queries are illegal while this thread captures a CUDA graph)
        if wait:
            self.event.synchronize()
        elif not self.event.query():
            return
        self.pending = False
        _StatusWatch._live.discard(self)
        code = int(self.pin[0])
        if code:
            self.pin[0] = 0
            raise EngineError("%s: tensor-core pipeline wait timed out (role code %d); the outputs of that call are "
                              "invalid" % (self.what, code))


def poll_status(wait=False):
    """Checks every status copy in flight (all modules, this process); ``wait=True`` blocks on the copies' events."""
    for w in list(_StatusWatch._live or ()):
        w.check(wait)


# ------------------------------------------------------------------------------------------
# Device-pointer path (what models.Generator.forward uses with torch tensors)
# ------------------------------------------------------------------------------------------
class GeneratorDevice:
    """Packed weights + workspace cache on one CUDA device, driven with torch tensors."""

    def __init__(self, device):
        import torch
        self.torch = torch
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise EngineError("the B200 engine runs on CUDA devices only (got %s)" % (device,))
        with torch.cuda.device(self.device):
            check(lib().mg_device_check())
        self.packed = torch.empty((lib().mg_gen_packed_bytes() + 3) // 4, dtype=torch.float32, device=self.device)
        self._ws = None
        self._ws_key = None
        self._watch = _StatusWatch(torch, self.device, "Generator.forward")

    def pack(self, vs, gs, bs):
        """vs/gs/bs: 30 contiguous fp32 CUDA tensors each (weight_v, weight_g, bias; reference order)."""
        torch = self.torch
        keep = []
        def ptrs(ts):
            out = []
            for t in ts:
                t = t.detach()
                if t.device != self.device or t.dtype != torch.float32:
                    raise EngineError("generator parameters must be fp32 tensors on %s" % (self.device,))
                t = t.contiguous()
                keep.append(t)
                out.append(t.data_ptr())
            return _ptr_array(out)
        if not (len(vs) == len(gs) == len(bs) == NUM_LAYERS):
            raise EngineError("expected %d layers" % NUM_LAYERS)
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            check(lib().mg_gen_pack(ptrs(vs), ptrs(gs), ptrs(bs), self.packed.data_ptr(), stream))
        del keep

    def workspace(self, B, T):
        need = lib().mg_gen_workspace_bytes(B, T)
        if self._ws is None or self._ws.numel() * 4 < need:
            self._ws = self.torch.empty((need + 3) // 4, dtype=self.torch.float32, device=self.device)
        return self._ws

    def forward(self, mel, out=None, lengths=None):
        """mel [B, 80, T] -> audio [B, 1, 256 T], asynchronous on the current stream.  lengths (optional, one value in [1, T]
        per item; see lengths_array): ragged batch -- item b is its first lengths[b] frames, its audio ends at 256 lengths[b]
        samples and is exactly zero after that (mg_gen_forward_varlen)."""
        torch = self.torch
        if mel.dim() != 3 or mel.shape[1] != 80:
            raise EngineError("mel must be [B, 80, T], got %s" % (tuple(mel.shape),))
        if mel.device != self.device or mel.dtype != torch.float32:
            raise EngineError("mel must be an fp32 tensor on %s" % (self.device,))
        mel = mel.contiguous()
        B, _, T = mel.shape
        lens = None if lengths is None else lengths_array(lengths, B)
        if out is None:
            out = torch.empty((B, 1, 256 * T), dtype=torch.float32, device=self.device)
        self._watch.check()  # the previous forward's status word, if its copy has landed
        ws = self.workspace(B, T)
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            if lens is None:
                check(lib().mg_gen_forward(self.packed.data_ptr(), mel.data_ptr(), out.data_ptr(), B, T,
                                           ws.data_ptr(), ws.numel() * 4, stream))
            else:
                check(lib().mg_gen_forward_varlen(self.packed.data_ptr(), mel.data_ptr(), out.data_ptr(), B, T, lens,
                                                  ws.data_ptr(), ws.numel() * 4, stream))
            off = (lib().mg_gen_workspace_bytes(B, T) - 256) // 4  # the status word sits after the activation buffers
            self._watch.arm(ws.view(torch.int32)[off:off + 1])
        return out

    def forward_timed(self, mel, out):
        """Like forward; returns {kernel name: device time in ms} for every launch of the forward."""
        torch = self.torch
        mel = mel.contiguous()
        B, _, T = mel.shape
        ws = self.workspace(B, T)
        n = lib().mg_gen_forward_launches()
        ms = (ctypes.c_float * 16)()
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            check(lib().mg_gen_forward_timed(self.packed.data_ptr(), mel.data_ptr(), out.data_ptr(), B, T,
                                             ws.data_ptr(), ws.numel() * 4, stream, ms))
        return [(lib().mg_gen_kernel_name(i).decode(), ms[i]) for i in range(n)]

    def check_status(self, B, T):
        """Synchronises and raises if the tensor-core pipeline of the last forward timed out."""
        torch = self.torch
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            check(lib().mg_gen_check_status(self._ws.data_ptr(), B, T, stream))

    def convt(self, stage, x):
        """LeakyReLU -> ConvTranspose1d of stage 0..3 on the tensor cores; x [B, 512>>stage, Lin]; synchronous."""
        torch = self.torch
        x = x.contiguous()
        B, C, L = x.shape
        if C != (512 >> stage):
            raise EngineError("stage %d expects %d input channels" % (stage, 512 >> stage))
        y = torch.empty((B, 256 >> stage, L * (8 if stage < 2 else 2)), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            check(lib().mg_gen_convt(self.packed.data_ptr(), stage, x.data_ptr(), y.data_ptr(), B, L, stream))
        return y

    def resblock(self, stage, x):
        """One tensor-core ResBlock (stage 0..3) on x [B, 256>>stage, L]; synchronous."""
        torch = self.torch
        x = x.contiguous()
        B, C, L = x.shape
        if C != (256 >> stage):
            raise EngineError("stage %d expects %d channels" % (stage, 256 >> stage))
        y = torch.empty_like(x)
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            check(lib().mg_gen_resblock(self.packed.data_ptr(), stage, x.data_ptr(), y.data_ptr(), B, L, stream))
        return y

    def upres(self, stage, x):
        """Stage 2 or 3 as one kernel: LeakyReLU -> ConvTranspose1d(k4, s2) -> ResBlock on x [B, 512>>stage, Lin];
        returns [B, 256>>stage, 2 Lin]; synchronous."""
        torch = self.torch
        x = x.contiguous()
        B, C, L = x.shape
        if stage not in (2, 3) or C != (512 >> stage):
            raise EngineError("upres: stage 2 / 3 expect 128 / 64 input channels")
        y = torch.empty((B, 256 >> stage, 2 * L), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            check(lib().mg_gen_upres(self.packed.data_ptr(), stage, x.data_ptr(), y.data_ptr(), B, L, stream))
        return y

    def resup(self, stage, x):
        """ResBlock `stage` (0..2) + the next stage's LeakyReLU -> ConvTranspose1d at its tail, one kernel:
        x [B, 256>>stage, L] -> [B, 128>>stage, S L] (S = 8 for stage 0, else 2); synchronous parity entry point."""
        torch = self.torch
        x = x.contiguous()
        B, C, L = x.shape
        if stage not in (0, 1, 2) or C != (256 >> stage):
            raise EngineError("resup: stage 0..2 with 256>>stage channels")
        y = torch.empty((B, C // 2, L * (8 if stage == 0 else 2)), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            check(lib().mg_gen_resup(self.packed.data_ptr(), stage, x.data_ptr(), y.data_ptr(), B, L, stream))
        return y

    def conv_pre(self, mel):
        """conv_pre alone (models.py:46,62): mel [B, 80, T] -> [B, 512, T]; synchronous parity entry point."""
        torch = self.torch
        mel = mel.contiguous()
        B, _, T = mel.shape
        y = torch.empty((B, 512, T), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            check(lib().mg_gen_conv_pre(self.packed.data_ptr(), mel.data_ptr(), y.data_ptr(), B, T, stream))
        return y

    def resblock_post(self, x):
        """Last ResBlock + LeakyReLU -> conv_post -> tanh (models.py:66-69) on x [B, 32, L] -> audio [B, 1, L]; synchronous."""
        torch = self.torch
        x = x.contiguous()
        B, C, L = x.shape
        if C != 32:
            raise EngineError("resblock_post expects 32 channels")
        y = torch.empty((B, 1, L), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            check(lib().mg_gen_resblock_post(self.packed.data_ptr(), x.data_ptr(), y.data_ptr(), B, L, stream))
        return y

    def stage_output(self, which, B, T):
        """Activation after conv_pre (0) or stage 0..2 (1..3) of the last forward, NCL."""
        torch = self.torch
        shapes = [(B, 512, T), (B, 256, 8 * T), (B, 128, 64 * T), (B, 64, 128 * T)]
        out = torch.empty(shapes[which], dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            check(lib().mg_gen_stage_output(self._ws.data_ptr(), which, out.data_ptr(), B, T, stream))
        return out


D_CHANNELS = (16, 64, 256, 1024, 1024, 1024, 1)  # channels of the seven feature maps of one Discriminator


def msd_lengths(L):
    """Feature-map lengths [3][7] of the multi-scale discriminator for an input of L samples."""
    lens = (ctypes.c_int * 21)()
    check(lib().mg_msd_lengths(int(L), lens))
    return [[lens[s * 7 + l] for l in range(7)] for s in range(3)]


LOSS_L1, LOSS_ONE_MINUS_SQ, LOSS_SQ = 0, 1, 2  # row modes of mg_loss_forward (include/melgan_b200.h)


def _loss_tables(a, b, modes):
    import torch
    dev = a[0].device
    if dev.type != "cuda":
        raise EngineError("the fused loss kernels run on CUDA tensors only")
    keep_a, keep_b = [], []
    for t, u, m in zip(a, b, modes):
        if t.dtype != torch.float32 or t.device != dev or (m == LOSS_L1 and (u is None or u.shape != t.shape or u.device != dev)):
            raise EngineError("loss rows must be fp32 tensors of equal shape on one CUDA device")
        keep_a.append(t.contiguous())
        keep_b.append(u.contiguous() if m == LOSS_L1 else None)
    n = (ctypes.c_longlong * len(a))(*[t.numel() for t in keep_a])
    md = (ctypes.c_int * len(a))(*modes)
    pa = _ptr_array([t.data_ptr() for t in keep_a])
    pb = _ptr_array([u.data_ptr() if u is not None else 0 for u in keep_b])
    return dev, keep_a, keep_b, n, md, pa, pb


def loss_forward(a, b, modes):
    """Row means of a fused loss table (mg_loss_forward): a, b lists of CUDA tensors, modes list of LOSS_*; returns a
    float32 CUDA tensor [len(a)].  One reduction launch + one fixed-order combine, no host sync."""
    import torch
    dev, keep_a, keep_b, n, md, pa, pb = _loss_tables(a, b, modes)
    out = torch.empty(len(a), dtype=torch.float32, device=dev)
    nbytes = lib().mg_loss_workspace_bytes(n, len(a))
    ws = torch.empty((nbytes + 3) // 4, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream().cuda_stream
        check(lib().mg_loss_forward(pa, pb, n, md, len(a), out.data_ptr(), ws.data_ptr(), nbytes, stream))
    return out


def loss_backward(a, b, modes, grad_out, need_b, out_a=None, out_b=None):
    """Gradients of the row means w.r.t. a (and b where need_b[i] and the row is an L1 pair), scaled by grad_out [rows].
    out_a / out_b: optional preallocated contiguous tensors to write into (e.g. the two halves of one stacked buffer)."""
    import torch
    dev, keep_a, keep_b, n, md, pa, pb = _loss_tables(a, b, modes)
    ga = list(out_a) if out_a is not None else [torch.empty_like(t) for t in keep_a]
    gb = (list(out_b) if out_b is not None else
          [torch.empty_like(u) if (u is not None and nb) else None for u, nb in zip(keep_b, need_b)])
    for t in ga + [u for u in gb if u is not None]:
        if not t.is_contiguous():
            raise EngineError("loss_backward: output gradients must be contiguous")
    pga = _ptr_array([t.data_ptr() for t in ga])
    pgb = _ptr_array([t.data_ptr() if t is not None else 0 for t in gb])
    grad_out = grad_out.to(device=dev, dtype=torch.float32).contiguous()
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream().cuda_stream
        check(lib().mg_loss_backward(pa, pb, n, md, len(a), grad_out.data_ptr(), pga, pgb, stream))
    return ga, gb


class DiscriminatorDevice:
    """Packed discriminator weights on one CUDA device, driven with torch tensors: the three-scale stack of
    MultiScaleDiscriminator (ndisc = 3) or one stand-alone Discriminator (ndisc = 1)."""

    def __init__(self, device, ndisc=3):
        import torch
        self.torch = torch
        self.device = torch.device(device)
        self.ndisc = ndisc
        if self.device.type != "cuda":
            raise EngineError("the B200 engine runs on CUDA devices only (got %s)" % (device,))
        if ndisc not in (1, 3):
            raise EngineError("DiscriminatorDevice: ndisc must be 1 or 3")
        with torch.cuda.device(self.device):
            check(lib().mg_device_check())
        nbytes = lib().mg_msd_packed_bytes() if ndisc == 3 else lib().mg_disc_packed_bytes()
        self.packed = torch.empty((nbytes + 3) // 4, dtype=torch.float32, device=self.device)
        self.status = torch.zeros(64, dtype=torch.int32, device=self.device)
        self._watch = _StatusWatch(torch, self.device, "Discriminator forward")

    def pack(self, vs, gs, bs):
        """vs/gs/bs: 7 * ndisc fp32 CUDA tensors each (discriminator-major, layers in registration order)."""
        torch = self.torch
        if not (len(vs) == len(gs) == len(bs) == 7 * self.ndisc):
            raise EngineError("expected %d discriminator layers" % (7 * self.ndisc))
        keep = []

        def ptrs(ts):
            out = []
            for t in ts:
                t = t.detach()
                if t.device != self.device or t.dtype != torch.float32:
                    raise EngineError("discriminator parameters must be fp32 tensors on %s" % (self.device,))
                t = t.contiguous()
                keep.append(t)
                out.append(t.data_ptr())
            return _ptr_array(out)
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            fn = lib().mg_msd_pack if self.ndisc == 3 else lib().mg_disc_pack
            check(fn(ptrs(vs), ptrs(gs), ptrs(bs), self.packed.data_ptr(), stream))

    def forward(self, y):
        """y [Bt, 1, L] -> list of ndisc lists of 7 feature maps [Bt, C, len] (fresh tensors)."""
        torch = self.torch
        if y.dim() != 3 or y.shape[1] != 1:
            raise EngineError("audio must be [B, 1, L], got %s" % (tuple(y.shape),))
        if y.device != self.device or y.dtype != torch.float32:
            raise EngineError("audio must be an fp32 tensor on %s" % (self.device,))
        y = y.contiguous()
        Bt, _, L = y.shape
        lens = msd_lengths(L)
        self._watch.check()
        fmaps = [[torch.empty((Bt, D_CHANNELS[l], lens[s][l]), dtype=torch.float32, device=self.device)
                  for l in range(7)] for s in range(self.ndisc)]
        ptrs = _ptr_array([f.data_ptr() for sc in fmaps for f in sc])
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            fn = lib().mg_msd_forward if self.ndisc == 3 else lib().mg_disc_forward
            check(fn(self.packed.data_ptr(), y.data_ptr(), Bt, L, ptrs, self.status.data_ptr(), stream))
            self._watch.arm(self.status[:1])
        return fmaps

    def scale_backward(self, scale, x0, fmaps, grads, need_gx0):
        """The whole backward of discriminator `scale` in one host call (mg_msd_scale_backward): x0 [Bt, 1, L0] its input,
        fmaps the 7 maps its forward returned, grads the gradient w.r.t. each (None: none).  Returns (gx0 | None, dws[7],
        dbs[7]) -- gradients of the FOLDED weights in torch layout; entries of layers the gradient does not reach are None.
        The intermediate gradients live in a workspace that is reused by every call on this device (the calls are ordered
        by the stream they are enqueued on)."""
        torch = self.torch
        from .synth import DISCRIMINATOR_LAYERS
        x0 = x0.contiguous()
        Bt, _, L0 = x0.shape
        gs = [g.contiguous() if g is not None else None for g in grads]
        keep = [f.contiguous() for f in fmaps]
        dws = [torch.empty((cout, cin // groups, k), dtype=torch.float32, device=self.device)
               for _n, cin, cout, k, _s, groups, _p in DISCRIMINATOR_LAYERS]
        dbs = [torch.empty((cout,), dtype=torch.float32, device=self.device) for _n, _cin, cout, *_ in DISCRIMINATOR_LAYERS]
        gx0 = torch.empty_like(x0) if need_gx0 else None
        nbytes = lib().mg_msd_scale_backward_workspace_bytes(Bt, L0)
        ws = self.__dict__.get("_bwd_ws")
        if ws is None or ws.numel() * 4 < nbytes:
            ws = self._bwd_ws = torch.empty((nbytes + 3) // 4, dtype=torch.float32, device=self.device)
        reached = (ctypes.c_int * 7)()
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            check(lib().mg_msd_scale_backward(
                self.packed.data_ptr(), scale, x0.data_ptr(), _ptr_array([f.data_ptr() for f in keep]),
                _ptr_array([g.data_ptr() if g is not None else None for g in gs]), gx0.data_ptr() if need_gx0 else None,
                _ptr_array([t.data_ptr() for t in dws]), _ptr_array([t.data_ptr() for t in dbs]), reached, ws.data_ptr(),
                ws.numel() * 4, Bt, L0, self.status.data_ptr(), stream))
        hit = [bool(r) for r in reached]
        return (gx0 if hit[0] else None), [w if h else None for w, h in zip(dws, hit)], [b if h else None for b, h in zip(dbs, hit)]

    def grouped_backward(self, scale, layer, dz, x, need_dx=True):
        """Gradients of grouped conv `layer` (1..4) of discriminator `scale`: dz [Bt, Cout, Lout] (already multiplied by
        LeakyReLU'), x [Bt, Cin, Lin] the layer input -> (dx or None, dw [Cout, 4, 41] w.r.t. the folded weight, db)."""
        torch = self.torch
        dz, x = dz.contiguous(), x.contiguous()
        Bt, cout, Lout = dz.shape
        _, cin, Lin = x.shape
        dx = torch.empty_like(x) if need_dx else None
        dw = torch.empty((cout, 4, 41), dtype=torch.float32, device=self.device)
        db = torch.empty(cout, dtype=torch.float32, device=self.device)
        nbytes = lib().mg_msd_grouped_backward_workspace_bytes(layer, Bt, Lout)
        ws = torch.empty((nbytes + 3) // 4, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            check(lib().mg_msd_grouped_backward(self.packed.data_ptr(), scale, layer, dz.data_ptr(), x.data_ptr(),
                                                dx.data_ptr() if need_dx else None, dw.data_ptr(), db.data_ptr(),
                                                ws.data_ptr(), nbytes, Bt, Lin, Lout, stream))
        return dx, dw, db

    def post1_dgrad(self, scale, dz):
        """dx of conv_post1 of discriminator `scale` from dz [Bt, 1024, L] (tcgen05, transposed weight copy of the blob)."""
        torch = self.torch
        dz = dz.contiguous()
        Bt, C, L = dz.shape
        if C != 1024:
            raise EngineError("post1_dgrad expects 1024 channels")
        dx = torch.empty_like(dz)
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            check(lib().mg_msd_post1_dgrad(self.packed.data_ptr(), scale, dz.data_ptr(), dx.data_ptr(), Bt, L,
                                           self.status.data_ptr(), stream))
        return dx

    def edge_backward(self, scale, layer, dz, x, need_dx=True):
        """(dx | None, dw, db) of conv_pre (layer 0) or conv_post2 (layer 6) of discriminator `scale`; dw in the torch layout."""
        torch = self.torch
        x, dz = x.contiguous(), dz.contiguous()
        Bt, L = x.shape[0], x.shape[2]
        cin, cout, k = (1, 16, 15) if layer == 0 else (1024, 1, 3)
        if tuple(x.shape) != (Bt, cin, L) or tuple(dz.shape) != (Bt, cout, L):
            raise EngineError(f"edge_backward(layer {layer}) expects x [Bt, {cin}, L] and dz [Bt, {cout}, L]")
        dx = torch.empty_like(x) if need_dx else None
        dw = torch.empty((cout, cin, k), dtype=torch.float32, device=x.device)
        db = torch.empty((cout,), dtype=torch.float32, device=x.device)
        nbytes = lib().mg_msd_edge_backward_workspace_bytes(layer, Bt, L)
        ws = torch.empty(max(nbytes // 4, 1), dtype=torch.float32, device=x.device)
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            check(lib().mg_msd_edge_backward(self.packed.data_ptr(), scale, layer, dz.data_ptr(), x.data_ptr(),
                                             dx.data_ptr() if need_dx else None, dw.data_ptr(), db.data_ptr(),
                                             ws.data_ptr(), nbytes, Bt, L, stream))
        return dx, dw, db

    def post1_wgrad(self, x, dz):
        """(dW [1024, 1024, 5], db [1024]) of conv_post1 from its input x and dz, both [Bt, 1024, L] (tcgen05, split-bf16)."""
        torch = self.torch
        x, dz = x.contiguous(), dz.contiguous()
        Bt, C, L = dz.shape
        if C != 1024 or tuple(x.shape) != (Bt, C, L):
            raise EngineError("post1_wgrad expects x and dz of shape [Bt, 1024, L]")
        dw = torch.empty((1024, 1024, 5), dtype=torch.float32, device=dz.device)
        db = torch.empty((1024,), dtype=torch.float32, device=dz.device)
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            check(lib().mg_msd_post1_wgrad(x.data_ptr(), dz.data_ptr(), dw.data_ptr(), db.data_ptr(), Bt, L,
                                           self.status.data_ptr(), stream))
        return dw, db

    def lrelu_backward(self, g1, g2, out):
        """(g1 + g2) * LeakyReLU'(out) in one launch; g1 or g2 may be None (not both)."""
        torch = self.torch
        if g1 is None:
            g1, g2 = g2, None
        g1 = g1.contiguous()
        g2 = g2.contiguous() if g2 is not None else None
        out = out.contiguous()
        dz = torch.empty_like(out)
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            check(lib().mg_lrelu_backward(g1.data_ptr(), g2.data_ptr() if g2 is not None else None, out.data_ptr(),
                                          dz.data_ptr(), out.numel(), stream))
        return dz

    def wn_backward(self, vs, gs, dws):
        """(d weight_v, d weight_g) of the 7 * ndisc layers from the gradients of their folded weights (None: layer skipped)."""
        torch = self.torch
        vs = [t.detach().contiguous() for t in vs]
        gs = [t.detach().contiguous() for t in gs]
        dws = [t.contiguous() if t is not None else None for t in dws]
        dvs = [torch.empty_like(v) if d is not None else None for v, d in zip(vs, dws)]
        dgs = [torch.empty_like(g) if d is not None else None for g, d in zip(gs, dws)]

        pad = 21 - len(vs)  # the launch walks a 21-row table; a stand-alone Discriminator fills the rest with skipped rows

        def arr(ts, fill):
            return _ptr_array([t.data_ptr() if t is not None else None for t in ts] + [fill] * pad)
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            check(lib().mg_msd_wn_backward(arr(vs, vs[0].data_ptr()), arr(gs, gs[0].data_ptr()), arr(dws, None), arr(dvs, None),
                                           arr(dgs, None), stream))
        return dvs, dgs

    def check_status(self):
        torch = self.torch
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            check(lib().mg_msd_check_status(self.status.data_ptr(), stream))


# ------------------------------------------------------------------------------------------
# Host-buffer path (no torch needed): numpy in, numpy out, copies inside the call
# ------------------------------------------------------------------------------------------
class GeneratorHost:
    """mg_gen_engine_* wrapper: the call a non-PyTorch host makes (host buffers in and out)."""

    def __init__(self, max_B=1, max_T=32):
        self._h = ctypes.c_void_p()
        check(lib().mg_gen_engine_create(ctypes.byref(self._h), max_B, max_T))

    def load_state(self, state):
        """state: mapping name -> float32 ndarray with the reference's state_dict keys."""
        from .synth import GENERATOR_LAYERS
        keep, vs, gs, bs = [], [], [], []
        for name, *_ in GENERATOR_LAYERS:
            for lst, suffix in ((vs, ".weight_v"), (gs, ".weight_g"), (bs, ".bias")):
                a = np.ascontiguousarray(state[name + suffix], dtype=np.float32)
                keep.append(a)
                lst.append(a.ctypes.data)
        check(lib().mg_gen_engine_load_state(self._h, _ptr_array(vs), _ptr_array(gs), _ptr_array(bs)))

    def forward(self, mel, out=None, lengths=None):
        """lengths (optional, one value in [1, T] per item): ragged batch, as GeneratorDevice.forward."""
        mel = np.ascontiguousarray(mel, dtype=np.float32)
        B, C, T = mel.shape
        if C != 80:
            raise EngineError("mel must be [B, 80, T]")
        if out is None:
            out = np.empty((B, 1, 256 * T), np.float32)
        if lengths is None:
            check(lib().mg_gen_engine_forward(self._h, mel.ctypes.data, out.ctypes.data, B, T))
        else:
            check(lib().mg_gen_engine_forward_varlen(self._h, mel.ctypes.data, out.ctypes.data, B, T, lengths_array(lengths, B)))
        return out

    def forward_ptr(self, mel_ptr, out_ptr, B, T):
        """Raw host pointers (e.g. pinned torch tensors' data_ptr())."""
        check(lib().mg_gen_engine_forward(self._h, mel_ptr, out_ptr, B, T))

    HALO_FRAMES = 8  # the generator's receptive field is +-7 mel frames (SURVEY section 5); 8 for slack

    def stream(self, mel, chunk_frames=128):
        """Long-utterance streaming (BASELINE config 5): yields the audio of `mel` [1, 80, T] chunk by chunk, each chunk
        computed from its frames plus an 8-frame halo either side, so latency and memory are bounded by the chunk and the
        concatenation equals the whole-utterance result (every conv of the fused stages re-applies its zero padding only
        at the true ends, which a chunk touching an end reproduces exactly)."""
        mel = np.ascontiguousarray(mel, dtype=np.float32)
        if mel.ndim != 3 or mel.shape[0] != 1 or mel.shape[1] != 80:
            raise EngineError("stream() takes one utterance [1, 80, T]")
        T, h = mel.shape[2], self.HALO_FRAMES
        for lo in range(0, T, chunk_frames):
            hi = min(T, lo + chunk_frames)
            a, b = max(0, lo - h), min(T, hi + h)
            audio = self.forward(mel[:, :, a:b])
            yield audio[:, :, (lo - a) * 256:(lo - a + hi - lo) * 256]

    def last_kernel_ms(self):
        ms = ctypes.c_float()
        check(lib().mg_gen_engine_last_kernel_ms(self._h, ctypes.byref(ms)))
        return ms.value

    def close(self):
        if self._h:
            lib().mg_gen_engine_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
