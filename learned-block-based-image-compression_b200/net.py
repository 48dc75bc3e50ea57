"""Host-side mirror of the reference model class for the codec path.

`BlockBasedImgCompLossyNetv9` keeps the method surface eval_model() uses on the reference model
(graphs/models/BlockBasedImgCompLossy_net.py:251-452, callers agents/blkbsdimgcomp_agent.py:555,
592, 598 and agents/base.py:95-96):

    Model(config)                      config.block_size / KS / N / M            NET:259-317
    .load_state_dict(sd)               the reference state_dict, verbatim          base.py:95-96
    .update(force=False) -> bool       entropy tables                              NET:121-125
    .compress(x, LRU, chlat)           -> (bytes, zhat)                            NET:319-361
    .decompress(bitstream, LRU, xshape, chlat, devc) -> zhat                       NET:400-452

plus batched, device-resident variants.  All arithmetic runs in liblbic_b200.so (sm_100a CUDA);
PyTorch only owns device memory and streams.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes
import math
from collections import OrderedDict
from types import SimpleNamespace

import numpy as np
import torch

from . import _lib
from .config import load_config
from .weights import layer_specs

SCALES_MIN, SCALES_MAX, SCALES_LEVELS = 0.11, 256, 64   # NET:13-15


def get_scale_table(mmin=SCALES_MIN, mmax=SCALES_MAX, levels=SCALES_LEVELS):
    """NET:17-18 (same torch expression, so the 64 fp32 thresholds are bit-identical)."""
    return torch.exp(torch.linspace(math.log(mmin), math.log(mmax), levels))


def get_lru(KS):
    """get_lru_(KS, 'compress') of the agent (AGENT:481-489)."""
    r = sum(int(k) // 2 for k in KS)
    return r, r, r


class BlockBasedImgCompLossyNetv9:
    def __init__(self, config, device=None):
        self.config = load_config(config)      # JSON path, built-in name, dict / EasyDict (the reference's config object), namespace
        c = self.config
        self.B, self.N, self.M = int(c.block_size), int(c.N), int(c.M)
        self.KS = [int(k) for k in c.KS]
        self.Cin = 3 * self.B * self.B
        self._sd = None
        self._handle = None
        self._device = None
        self._tables_ready = False
        self.conditional_gaussian_model = SimpleNamespace(
            quantized_cdf=torch.IntTensor(), cdf_length=torch.IntTensor(), offset=torch.IntTensor(),
            scale_table=torch.Tensor(), tail_mass=1e-9)
        self.training = False
        if device is not None:
            self.to(device)

    # ---- nn.Module-like plumbing ------------------------------------------------------------
    def eval(self):
        self.training = False
        return self

    def to(self, device):
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("lbic_b200 runs on sm_100a GPUs only; there is no CPU path")
        idx = device.index if device.index is not None else torch.cuda.current_device()
        if self._handle is not None and self._device.index == idx:
            return self
        self._destroy()
        L = _lib.lib()
        cfg = _lib.LbicConfig(self.B, (ctypes.c_int * 4)(*self.KS), self.N, self.M)
        h = ctypes.c_void_p()
        _lib.check(L.lbic_create(ctypes.byref(cfg), idx, ctypes.byref(h)))
        self._handle, self._device = h, torch.device("cuda", idx)
        if self._sd is not None:
            self._upload()
        return self

    def cuda(self, device=None):
        return self.to(torch.device("cuda", torch.cuda.current_device() if device is None else device))

    def _destroy(self):
        if self._handle is not None:
            _lib.lib().lbic_destroy(self._handle)
            self._handle = None
            self._tables_ready = False

    def __del__(self):
        try:
            self._destroy()
        except Exception:
            pass

    def _need(self):
        if self._handle is None:
            if torch.cuda.is_available():
                self.to(torch.device("cuda", torch.cuda.current_device()))
            else:
                raise RuntimeError("lbic_b200: no CUDA device; the B200 path has no CPU fallback")
        return self._handle

    def _stream(self):
        return torch.cuda.current_stream(self._device).cuda_stream

    def set_gemm_core(self, core: str):
        """'tcgen05' (product path) or 'simt' (fp32 cross-check twin)."""
        _lib.check(_lib.lib().lbic_set_option(self._need(), _lib.LBIC_OPT_GEMM_CORE, {"tcgen05": 0, "simt": 1}[core]))

    def set_option(self, name: str, value: int):
        """Tuning hooks: 'force_bn' (forced tile width), 'ws' (0 off / 1 auto / 2 always: persistent kernel),
        'pair' (CTA-pair form of the persistent kernel), 'pdl', 'host_bands' (bands of block rows of the host calls),
        'wave' (persistent wavefront kernel for small steps), 'wave_max_rows'."""
        opt = {"force_bn": _lib.LBIC_OPT_FORCE_BN, "wave": _lib.LBIC_OPT_WAVE, "wave_max_rows": _lib.LBIC_OPT_WAVE_MAX_ROWS, "wave_dec_max_rows": _lib.LBIC_OPT_WAVE_DEC_MAX_ROWS,
               "wave_bn": _lib.LBIC_OPT_WAVE_BN, "dec_smem_warp": _lib.LBIC_OPT_DEC_SMEM_WARP, "check_saturation": _lib.LBIC_OPT_CHECK_SATURATION, "flow_pair_min_rows": _lib.LBIC_OPT_FLOW_PAIR_MIN_ROWS,
               "ws": _lib.LBIC_OPT_WS, "pdl": _lib.LBIC_OPT_PDL,
               "pair": _lib.LBIC_OPT_PAIR, "dec_thread_rows": _lib.LBIC_OPT_DEC_THREAD_ROWS,
               "enc_thread_streams": _lib.LBIC_OPT_ENC_THREAD_STREAMS, "enc_block_streams": _lib.LBIC_OPT_ENC_BLOCK_STREAMS, "flow": _lib.LBIC_OPT_FLOW,
               "flow_min_rows": _lib.LBIC_OPT_FLOW_MIN_ROWS,
               "host_bands": _lib.LBIC_OPT_HOST_BANDS}[name]
        _lib.check(_lib.lib().lbic_set_option(self._need(), opt, int(value)))

    # ---- state_dict ----------------------------------------------------------------------------
    def expected_keys(self):
        keys = []
        for prefix, kind, _ in layer_specs(self.config):
            if kind == "conv":
                keys += [prefix + s for s in (".weight", ".bias", ".mask")]
            else:
                keys += [prefix + s for s in (".beta", ".gamma", ".beta_reparam.pedestal",
                                              ".beta_reparam.lower_bound.bound", ".gamma_reparam.pedestal",
                                              ".gamma_reparam.lower_bound.bound")]
        return keys

    def load_state_dict(self, state_dict, strict: bool = True):
        """Accepts the reference `state_dict0` verbatim (SURVEY.md Appendix A.7).  Keys under
        conditional_gaussian_model.* are optional (they are empty in released checkpoints, AGENT:570);
        non-empty table buffers are installed instead of being rebuilt."""
        need = self.expected_keys()
        missing = [k for k in need if k not in state_dict and not k.endswith(".mask") and "reparam" not in k]
        if missing:
            raise RuntimeError(f"Missing key(s) in state_dict: {missing[:6]}{' ...' if len(missing) > 6 else ''}")
        if strict:
            extra = [k for k in state_dict if k not in need and not k.startswith("conditional_gaussian_model.")]
            if extra:
                raise RuntimeError(f"Unexpected key(s) in state_dict: {extra[:6]}")
        self._sd = OrderedDict((k, v.detach().clone()) for k, v in state_dict.items())
        if self._handle is not None:
            self._upload()
        cg = "conditional_gaussian_model."
        q = self._sd.get(cg + "_quantized_cdf")
        if q is not None and q.numel() > 0:
            self.conditional_gaussian_model.quantized_cdf = q.int().cpu()
            self.conditional_gaussian_model.cdf_length = self._sd[cg + "_cdf_length"].int().cpu()
            self.conditional_gaussian_model.offset = self._sd[cg + "_offset"].int().cpu()
            st = self._sd.get(cg + "scale_table")
            self.conditional_gaussian_model.scale_table = (st.float().cpu() if st is not None and st.numel() == 64
                                                           else get_scale_table())
            self._tables_ready = False
            if self._handle is not None:
                self._install_tables()
        return SimpleNamespace(missing_keys=[], unexpected_keys=[])

    def state_dict(self):
        sd = OrderedDict(self._sd or {})
        g = self.conditional_gaussian_model
        sd["conditional_gaussian_model._offset"] = g.offset
        sd["conditional_gaussian_model._quantized_cdf"] = g.quantized_cdf
        sd["conditional_gaussian_model._cdf_length"] = g.cdf_length
        sd["conditional_gaussian_model.scale_table"] = g.scale_table
        return sd

    def _upload(self):
        L = _lib.lib()
        keep, descs = [], []
        for k, v in self._sd.items():
            if k.startswith("conditional_gaussian_model.") or not v.dtype.is_floating_point or v.numel() == 0:
                continue
            t = v.detach().to(torch.float32).contiguous()
            keep.append(t)
            d = _lib.LbicTensorDesc()
            d.name = k.encode()
            d.data = t.data_ptr()
            d.ndim = t.dim()
            for i, s in enumerate(t.shape[:4]):
                d.shape[i] = s
            descs.append(d)
        arr = (_lib.LbicTensorDesc * len(descs))(*descs)
        with torch.cuda.device(self._device):
            _lib.check(L.lbic_load_weights(self._handle, arr, len(descs), self._stream()))
        if self.conditional_gaussian_model.quantized_cdf.numel() > 0 and not self._tables_ready:
            self._install_tables()

    # ---- entropy tables -------------------------------------------------------------------------
    def _install_tables(self):
        g = self.conditional_gaussian_model
        cdf = np.ascontiguousarray(g.quantized_cdf.numpy().astype(np.int32))
        ln = np.ascontiguousarray(g.cdf_length.numpy().astype(np.int32))
        off = np.ascontiguousarray(g.offset.numpy().astype(np.int32))
        st = np.ascontiguousarray(g.scale_table.numpy().astype(np.float32))
        _lib.check(_lib.lib().lbic_set_tables(self._need(), st.ctypes.data, 64, cdf.ctypes.data, cdf.shape[1],
                                              ln.ctypes.data, off.ctypes.data))
        self._tables_ready = True

    def update(self, force: bool = False) -> bool:
        """NET:121-125 -> GaussianConditional.update_scale_table (ENT:579-588): rebuilds the quantised
        CDF / cdf_length / offset tables, on the GPU.  Returns True if the tables were (re)built."""
        h = self._need()
        g = self.conditional_gaussian_model
        if g.offset.numel() > 0 and not force:
            if not self._tables_ready:
                self._install_tables()
            return False
        st = get_scale_table().contiguous()
        with torch.cuda.device(self._device):
            _lib.check(_lib.lib().lbic_build_tables(h, st.data_ptr(), 64, float(g.tail_mass), self._stream()))
        n, stride = ctypes.c_int(), ctypes.c_int()
        _lib.check(_lib.lib().lbic_get_tables(h, ctypes.byref(n), ctypes.byref(stride), None, None, None))
        cdf = np.empty((n.value, stride.value), dtype=np.int32)
        ln = np.empty(n.value, dtype=np.int32)
        off = np.empty(n.value, dtype=np.int32)
        _lib.check(_lib.lib().lbic_get_tables(h, None, None, cdf.ctypes.data, ln.ctypes.data, off.ctypes.data))
        g.quantized_cdf, g.cdf_length, g.offset = torch.from_numpy(cdf), torch.from_numpy(ln), torch.from_numpy(off)
        g.scale_table = st
        self._tables_ready = True
        return True

    # ---- codec path -------------------------------------------------------------------------------
    def _check_call(self, LRU, chlat):
        if LRU is not None and [int(v) for v in LRU] != list(get_lru(self.KS)):
            raise ValueError(f"LRU {list(LRU)} does not match KS {self.KS} (expected {list(get_lru(self.KS))})")
        if chlat is not None and int(chlat) != self.M:
            raise ValueError(f"chlat {chlat} != config.M {self.M}")

    def stream_bound(self, Hb, Wb, lanes=1):
        return int(_lib.lib().lbic_stream_bound(self._need(), Hb, Wb, lanes))

    def encode_device(self, x, lanes: int = 1, want_symbols: bool = False, entropy_code: bool = True,
                      stream_cap: int | None = None, out=None):
        """Batched encode with everything left on the device (no host synchronisation).
        x: (n, 3B^2, Hb, Wb) fp32 CUDA tensor in [-0.5, 0.5].
        Returns a namespace: zhat (n,3B^2,Hb,Wb), streams (n, cap) uint8, lens (n,) int32 [bytes],
        and sym (n,Hb,Wb,M) int32 / idx uint8 when want_symbols."""
        h = self._need()
        if not (x.is_cuda and x.dtype == torch.float32 and x.dim() == 4 and x.shape[1] == self.Cin):
            raise ValueError(f"x must be a CUDA fp32 tensor of shape (n, {self.Cin}, Hb, Wb)")
        x = x.contiguous()
        n, _, Hb, Wb = x.shape
        dev = x.device
        o = out if out is not None else SimpleNamespace()
        if out is None:
            o.zhat = torch.empty_like(x)
            o.sym = torch.empty(n, Hb, Wb, self.M, dtype=torch.int32, device=dev) if want_symbols else None
            o.idx = torch.empty(n, Hb, Wb, self.M, dtype=torch.uint8, device=dev) if want_symbols else None
            if entropy_code:
                cap = stream_cap or self.stream_bound(Hb, Wb, lanes)
                cap = (cap + 3) // 4 * 4
                o.streams = torch.empty(n, cap, dtype=torch.uint8, device=dev)
                o.lens = torch.zeros(n, dtype=torch.int32, device=dev)
            else:
                o.streams, o.lens = None, None
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().lbic_encode(
                h, x.data_ptr(), n, Hb, Wb, o.zhat.data_ptr(),
                o.sym.data_ptr() if o.sym is not None else None,
                o.idx.data_ptr() if o.idx is not None else None,
                o.streams.data_ptr() if o.streams is not None else None,
                o.streams.shape[1] if o.streams is not None else 0,
                o.lens.data_ptr() if o.lens is not None else None, lanes, self._stream()))
        return o

    def encode_device_mixed(self, xs, lanes: int = 1, want_symbols: bool = False, stream_cap: int | None = None):
        """One encode of differently sized images (lbic_encode_mixed); each image comes out exactly as encode_device of
        it alone.  xs: list of (1, 3B^2, Hb_i, Wb_i) or (3B^2, Hb_i, Wb_i) fp32 CUDA tensors on one device.  Returns a
        namespace: zhat / sym / idx (lists of per-image views of the packed outputs), streams (n, cap) uint8, lens (n,)
        int32, shapes [(Hb_i, Wb_i)]; no host synchronisation."""
        h = self._need()
        xs = [x[0] if x.dim() == 4 and x.shape[0] == 1 else x for x in xs]
        if not xs or any(not (x.is_cuda and x.dtype == torch.float32 and x.dim() == 3 and x.shape[0] == self.Cin) for x in xs):
            raise ValueError(f"xs must be a non-empty list of CUDA fp32 tensors of shape (1, {self.Cin}, Hb, Wb)")
        dev = xs[0].device
        shapes = [(int(x.shape[1]), int(x.shape[2])) for x in xs]
        n, counts = len(xs), [hb * wb for hb, wb in shapes]
        x = torch.cat([t.reshape(-1) for t in xs]).to(dev)
        o = SimpleNamespace(shapes=shapes)
        zhat = torch.empty_like(x)
        total = sum(counts)
        sym = torch.empty(total * self.M, dtype=torch.int32, device=dev) if want_symbols else None
        idx = torch.empty(total * self.M, dtype=torch.uint8, device=dev) if want_symbols else None
        cap = stream_cap or max(self.stream_bound(hb, wb, lanes) for hb, wb in shapes)
        cap = (cap + 3) // 4 * 4
        o.streams = torch.empty(n, cap, dtype=torch.uint8, device=dev)
        o.lens = torch.zeros(n, dtype=torch.int32, device=dev)
        Hb = (ctypes.c_int * n)(*[s[0] for s in shapes])
        Wb = (ctypes.c_int * n)(*[s[1] for s in shapes])
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().lbic_encode_mixed(
                h, x.data_ptr(), n, Hb, Wb, zhat.data_ptr(), sym.data_ptr() if sym is not None else None,
                idx.data_ptr() if idx is not None else None, o.streams.data_ptr(), cap, o.lens.data_ptr(), lanes,
                self._stream()))
        o.zhat = self._split(zhat, shapes, lambda hb, wb: (1, self.Cin, hb, wb), self.Cin)
        o.sym = self._split(sym, shapes, lambda hb, wb: (1, hb, wb, self.M), self.M) if sym is not None else None
        o.idx = self._split(idx, shapes, lambda hb, wb: (1, hb, wb, self.M), self.M) if idx is not None else None
        return o

    @staticmethod
    def _split(flat, shapes, shape_of, per_block):
        out, at = [], 0
        for hb, wb in shapes:
            k = hb * wb * per_block
            out.append(flat[at: at + k].view(*shape_of(hb, wb)))
            at += k
        return out

    def decode_device_mixed(self, streams, lens, shapes, lanes: int = 1, want_symbols: bool = False):
        """streams (n, cap) uint8 CUDA, lens (n,) int32 CUDA, shapes [(Hb_i, Wb_i)] -> list of zhat (1, 3B^2, Hb_i, Wb_i)
        [, list of sym (1, Hb_i, Wb_i, M)] (lbic_decode_mixed).  Asynchronous like decode_device."""
        h = self._need()
        dev = streams.device
        shapes = [(int(a), int(b)) for a, b in shapes]
        n, total = len(shapes), sum(a * b for a, b in shapes)
        zhat = torch.empty(total * self.Cin, dtype=torch.float32, device=dev)
        sym = torch.empty(total * self.M, dtype=torch.int32, device=dev) if want_symbols else None
        Hb = (ctypes.c_int * n)(*[s[0] for s in shapes])
        Wb = (ctypes.c_int * n)(*[s[1] for s in shapes])
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().lbic_decode_mixed(h, streams.data_ptr(), lens.data_ptr(), streams.shape[1], n, Hb, Wb,
                                                    zhat.data_ptr(), sym.data_ptr() if sym is not None else None, lanes,
                                                    self._stream()))
        z = self._split(zhat, shapes, lambda hb, wb: (1, self.Cin, hb, wb), self.Cin)
        if want_symbols:
            return z, self._split(sym, shapes, lambda hb, wb: (1, hb, wb, self.M), self.M)
        return z

    def validate_recu_reco(self, x):
        """Closed loop without entropy coding + rate estimate (validate_recu_reco_fast, AGENT:491-549).
        x: (n, 3B^2, Hb, Wb) CUDA fp32 -> (zhat, self_infos (n, M, Hb, Wb)); rate as the reference's loss computes it
        (graphs/losses/rate_dist.py:44): self_infos.sum() / x.numel() * 3  [bits per pixel]."""
        h = self._need()
        x = x.contiguous()
        n, _, Hb, Wb = x.shape
        zhat = torch.empty_like(x)
        info = torch.empty(n, self.M, Hb, Wb, dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            _lib.check(_lib.lib().lbic_validate(h, x.data_ptr(), n, Hb, Wb, zhat.data_ptr(), info.data_ptr(),
                                                self._stream()))
        return zhat, info

    def forward(self, zhat, x, clamp: bool = False, return_symbols: bool = False):
        """model.forward(zhat, x) of the reference in eval mode (NET:90-106): open-loop pass over every block given
        the context reconstruction zhat.  Both (n, 3B^2, Hb, Wb) CUDA fp32 -> (xhat, self_informations (n, M, Hb, Wb))
        [+ symbols (n, Hb, Wb, M)].  xhat is returned unclamped like the reference's; clamp=True applies the caller's
        clamp_(-0.5, 0.5) (AGENT:667) in the kernel."""
        h = self._need()
        if not (x.is_cuda and zhat.is_cuda and x.dtype == torch.float32 and zhat.dtype == torch.float32
                and x.dim() == 4 and x.shape[1] == self.Cin and zhat.shape == x.shape):
            raise ValueError(f"zhat and x must be CUDA fp32 tensors of the same shape (n, {self.Cin}, Hb, Wb)")
        x, zhat = x.contiguous(), zhat.contiguous()
        n, _, Hb, Wb = x.shape
        xhat = torch.empty_like(x)
        info = torch.empty(n, self.M, Hb, Wb, dtype=torch.float32, device=x.device)
        sym = torch.empty(n, Hb, Wb, self.M, dtype=torch.int32, device=x.device) if return_symbols else None
        with torch.cuda.device(x.device):
            _lib.check(_lib.lib().lbic_forward(h, zhat.data_ptr(), x.data_ptr(), n, Hb, Wb, xhat.data_ptr(),
                                               info.data_ptr(), sym.data_ptr() if sym is not None else None,
                                               1 if clamp else 0, self._stream()))
        return (xhat, info, sym) if return_symbols else (xhat, info)

    __call__ = forward

    def check_errors(self):
        """Synchronises the current stream and raises if the last encode / decode enqueued on it flagged an overflowing
        stream buffer (RuntimeError) or a malformed lane container (RuntimeError, 'malformed')."""
        with torch.cuda.device(self._device):
            _lib.check(_lib.lib().lbic_check_errors(self._need(), self._stream()))

    def decode_device(self, streams, lens, n, Hb, Wb, lanes: int = 1, want_symbols: bool = False):
        """streams (n, cap) uint8 CUDA, lens (n,) int32 CUDA -> zhat (n,3B^2,Hb,Wb) [, sym].  Asynchronous: a malformed
        lane container is only flagged on the device; call check_errors() (decompress_batch does)."""
        h = self._need()
        dev = streams.device
        zhat = torch.empty(n, self.Cin, Hb, Wb, dtype=torch.float32, device=dev)
        sym = torch.empty(n, Hb, Wb, self.M, dtype=torch.int32, device=dev) if want_symbols else None
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().lbic_decode(h, streams.data_ptr(), lens.data_ptr(), streams.shape[1], n, Hb, Wb,
                                              zhat.data_ptr(), sym.data_ptr() if sym is not None else None, lanes,
                                              self._stream()))
        return (zhat, sym) if want_symbols else zhat

    @staticmethod
    def _gather_streams(o):
        lens = o.lens.cpu().numpy().astype(np.int64)
        if (lens < 0).any() or (lens > o.streams.shape[1]).any():
            raise RuntimeError("bitstream buffer overflow (stream_cap too small)")
        host = o.streams[:, : int(lens.max())].cpu().numpy()
        return [host[i, : lens[i]].tobytes() for i in range(len(lens))]

    def compress_batch(self, x, lanes: int = 1, return_symbols: bool = False):
        """-> (list[bytes], zhat) or (list[bytes], zhat, sym, idx).  x: a (n, 3B^2, Hb, Wb) tensor, or a list of
        differently sized (1, 3B^2, Hb_i, Wb_i) tensors (one mixed-size call; zhat / sym / idx are then lists)."""
        if isinstance(x, (list, tuple)):
            o = self.encode_device_mixed(list(x), lanes=lanes, want_symbols=return_symbols)
        else:
            o = self.encode_device(x, lanes=lanes, want_symbols=return_symbols)
        strings = self._gather_streams(o)
        return (strings, o.zhat, o.sym, o.idx) if return_symbols else (strings, o.zhat)

    def decompress_batch(self, strings, xshape, lanes: int = 1, device=None):
        """xshape: (n, 3B^2, Hb, Wb) for n images of one size, or a list of per-image shapes ((1, 3B^2, Hb_i, Wb_i) or
        (Hb_i, Wb_i)) for one mixed-size call, which returns a list of zhat tensors."""
        self._need()
        dev = torch.device(device) if device is not None else self._device
        if isinstance(xshape, (list, tuple)) and len(xshape) > 0 and isinstance(xshape[0], (list, tuple, torch.Size)):
            shapes = [tuple(int(v) for v in s)[-2:] for s in xshape]
            if len(strings) != len(shapes) or any(len(s) == 4 and int(s[1]) != self.Cin for s in xshape):
                raise ValueError("strings / xshape mismatch")
            cap = (max(len(s) for s in strings) + 3) // 4 * 4
            host = np.zeros((len(strings), cap), dtype=np.uint8)
            for i, s in enumerate(strings):
                host[i, : len(s)] = np.frombuffer(s, dtype=np.uint8)
            lens = torch.tensor([len(s) for s in strings], dtype=torch.int32, device=dev)
            zs = self.decode_device_mixed(torch.from_numpy(host).to(dev), lens, shapes, lanes=lanes)
            self.check_errors()
            return zs
        n, ch, Hb, Wb = [int(v) for v in xshape]
        if len(strings) != n or ch != self.Cin:
            raise ValueError("strings / xshape mismatch")
        cap = (max(len(s) for s in strings) + 3) // 4 * 4
        host = np.zeros((n, cap), dtype=np.uint8)
        for i, s in enumerate(strings):
            host[i, : len(s)] = np.frombuffer(s, dtype=np.uint8)
        streams = torch.from_numpy(host).to(dev)
        lens = torch.tensor([len(s) for s in strings], dtype=torch.int32, device=dev)
        zhat = self.decode_device(streams, lens, n, Hb, Wb, lanes=lanes)
        self.check_errors()
        return zhat

    # ---- 8-bit images in host memory (eval_model's per-image body for a batch, AGENT:581-599, 610-628) -------------
    def compress_images_u8(self, images, lanes: int = 1, return_recon: bool = False, stream_cap: int | None = None):
        """images: (n, 3, H, W) uint8, host (numpy array or CPU tensor; pinned memory makes the copies asynchronous).
        -> (list[bytes], recon uint8 (n,3,H,W) or None).  ToTensor, -0.5, replicate padding, space-to-depth, compress
        and (optionally) the 8-bit reconstruction the reference would save, in one call."""
        h = self._need()
        a = images.numpy() if isinstance(images, torch.Tensor) else np.ascontiguousarray(images)
        if a.dtype != np.uint8 or a.ndim != 4 or a.shape[1] != 3:
            raise ValueError("images must be uint8 of shape (n, 3, H, W)")
        n, _, H, W = a.shape
        Hb, Wb = -(-H // self.B), -(-W // self.B)
        cap = (int(stream_cap or self.stream_bound(Hb, Wb, lanes)) + 3) // 4 * 4
        streams = np.empty((n, cap), dtype=np.uint8)
        lens = np.zeros(n, dtype=np.uint32)
        recon = np.empty_like(a) if return_recon else None
        with torch.cuda.device(self._device):
            _lib.check(_lib.lib().lbic_encode_images_u8_host(
                h, a.ctypes.data, n, H, W, recon.ctypes.data if recon is not None else None, streams.ctypes.data, cap,
                lens.ctypes.data, lanes))
        return [streams[i, : lens[i]].tobytes() for i in range(n)], recon

    def decompress_images_u8(self, strings, H: int, W: int, lanes: int = 1):
        """list[bytes] -> (n, 3, H, W) uint8 numpy array: decompress + depth-to-space + crop + 8-bit quantisation."""
        h = self._need()
        n = len(strings)
        cap = (max(len(s) for s in strings) + 3) // 4 * 4
        host = np.zeros((n, cap), dtype=np.uint8)
        for i, s in enumerate(strings):
            host[i, : len(s)] = np.frombuffer(s, dtype=np.uint8)
        lens = np.array([len(s) for s in strings], dtype=np.uint32)
        out = np.empty((n, 3, H, W), dtype=np.uint8)
        with torch.cuda.device(self._device):
            _lib.check(_lib.lib().lbic_decode_images_u8_host(h, host.ctypes.data, lens.ctypes.data, cap, n, H, W,
                                                             out.ctypes.data, lanes))
        return out

    # ---- 8-bit images of different sizes (lbic_encode_images_u8_host_mixed / lbic_decode_images_u8_host_mixed) ----
    def _pinned(self, name, nbytes):
        """Grow-only pinned host staging buffer (uint8), so that the call's band copies are asynchronous."""
        buf = getattr(self, name, None)
        if buf is None or buf.numel() < nbytes:
            buf = torch.empty(max(int(nbytes), 1), dtype=torch.uint8, pin_memory=True)
            setattr(self, name, buf)
        return buf

    def _pack_u8(self, images, hwc):
        """images -> (pinned packed (3, H_i, W_i) planes, [(H_i, W_i)]); hwc: (H, W, 3) arrays, transposed while packing."""
        arrs = [im.numpy() if isinstance(im, torch.Tensor) else np.asarray(im) for im in images]
        if not arrs or any(a.dtype != np.uint8 or a.ndim != 3 or a.shape[2 if hwc else 0] != 3 for a in arrs):
            raise ValueError("images must be a non-empty list of uint8 arrays of shape " + ("(H, W, 3)" if hwc else "(3, H, W)"))
        sizes = [(int(a.shape[0]), int(a.shape[1])) if hwc else (int(a.shape[1]), int(a.shape[2])) for a in arrs]
        total = sum(3 * H * W for H, W in sizes)
        buf = self._pinned("_pin_in", total)
        at = 0
        for a, (H, W) in zip(arrs, sizes):
            t = torch.from_numpy(np.ascontiguousarray(a))
            buf[at: at + 3 * H * W].view(3, H, W).copy_(t.permute(2, 0, 1) if hwc else t)
            at += 3 * H * W
        return buf, sizes

    def _unpack_u8(self, buf, sizes):
        out, at = [], 0
        for H, W in sizes:
            out.append(buf[at: at + 3 * H * W].view(3, H, W).numpy().copy())
            at += 3 * H * W
        return out

    def _compress_u8_mixed(self, images, hwc, lanes=1, return_recon=False, stream_cap=None):
        h = self._need()
        buf, sizes = self._pack_u8(images, hwc)
        n = len(sizes)
        grids = [(-(-H // self.B), -(-W // self.B)) for H, W in sizes]
        cap = (int(stream_cap or max(self.stream_bound(hb, wb, lanes) for hb, wb in grids)) + 3) // 4 * 4
        streams = np.empty((n, cap), dtype=np.uint8)
        lens = np.zeros(n, dtype=np.uint32)
        rec = self._pinned("_pin_out", sum(3 * H * W for H, W in sizes)) if return_recon else None
        Hs = (ctypes.c_int * n)(*[s[0] for s in sizes])
        Ws = (ctypes.c_int * n)(*[s[1] for s in sizes])
        with torch.cuda.device(self._device):
            _lib.check(_lib.lib().lbic_encode_images_u8_host_mixed(
                h, buf.data_ptr(), n, Hs, Ws, rec.data_ptr() if rec is not None else None, streams.ctypes.data, cap,
                lens.ctypes.data, lanes))
        return [streams[i, : lens[i]].tobytes() for i in range(n)], (self._unpack_u8(rec, sizes) if return_recon else None)

    def compress_images_u8_mixed(self, images, lanes: int = 1, return_recon: bool = False, stream_cap: int | None = None):
        """images: list of (3, H_i, W_i) uint8 numpy arrays or CPU tensors of any sizes -> (list[bytes], list of
        (3, H_i, W_i) uint8 reconstructions or None), in one call (lbic_encode_images_u8_host_mixed).  Each image comes
        out exactly as compress_images_u8 of that image alone.  The images are packed into a pinned staging buffer."""
        return self._compress_u8_mixed(images, False, lanes, return_recon, stream_cap)

    def decompress_images_u8_mixed(self, strings, sizes, lanes: int = 1):
        """list[bytes], [(H_i, W_i)] -> list of (3, H_i, W_i) uint8 arrays, in one call; each equals
        decompress_images_u8 of that stream alone."""
        h = self._need()
        sizes = [(int(a), int(b)) for a, b in sizes]
        n = len(strings)
        if n == 0 or len(sizes) != n:
            raise ValueError("strings / sizes mismatch")
        cap = (max(len(s) for s in strings) + 3) // 4 * 4
        host = np.zeros((n, max(cap, 4)), dtype=np.uint8)
        for i, s in enumerate(strings):
            host[i, : len(s)] = np.frombuffer(s, dtype=np.uint8)
        lens = np.array([len(s) for s in strings], dtype=np.uint32)
        out = self._pinned("_pin_out", sum(3 * H * W for H, W in sizes))
        Hs = (ctypes.c_int * n)(*[s[0] for s in sizes])
        Ws = (ctypes.c_int * n)(*[s[1] for s in sizes])
        with torch.cuda.device(self._device):
            _lib.check(_lib.lib().lbic_decode_images_u8_host_mixed(h, host.ctypes.data, lens.ctypes.data, host.shape[1], n,
                                                                   Hs, Ws, out.data_ptr(), lanes))
        return self._unpack_u8(out, sizes)

    def compress(self, x, LRU=None, chlat=None):
        """NET:319-361: one image (1, 3B^2, Hb, Wb) -> (bitstream bytes, zhat)."""
        self._check_call(LRU, chlat)
        if x.shape[0] != 1:
            raise ValueError("compress() takes one image; use compress_batch() for more")
        strings, zhat = self.compress_batch(x, lanes=1)
        return strings[0], zhat

    def decompress(self, bitstream, LRU=None, xshape=None, chlat=None, devc=None):
        """NET:400-452: bitstream bytes -> zhat (1, 3B^2, Hb, Wb)."""
        self._check_call(LRU, chlat)
        return self.decompress_batch([bitstream], xshape, lanes=1, device=devc)

    # ---- quality figures of eval_model, on the GPU (AGENT:611-619) -------------------------------------------------
    def image_metrics(self, x, y, msssim: bool = True, offset: float = 0.5, data_range: float = 1.0):
        """x, y: (n, C, H, W) CUDA fp32 images (eval_model passes the [-0.5, 0.5] original and reconstruction).
        -> dict(mse=[n], psnr=[n], msssim=[n] or None): mse = F.mse_loss per image, psnr = -10 log10(mse),
        msssim = pytorch_msssim.ms_ssim(x + offset, y + offset, data_range) per image."""
        if not (x.is_cuda and y.is_cuda and x.shape == y.shape and x.dim() == 4 and x.dtype == torch.float32 == y.dtype):
            raise ValueError("x and y must be CUDA fp32 tensors of the same (n, C, H, W) shape")
        x, y = x.contiguous(), y.contiguous()
        n, C, H, W = x.shape
        mse = np.zeros(n, dtype=np.float64)
        ms = np.zeros(n, dtype=np.float64) if msssim else None
        with torch.cuda.device(x.device):
            _lib.check(_lib.lib().lbic_image_metrics(self._need(), x.data_ptr(), y.data_ptr(), n, C, H, W, float(offset),
                                                     float(data_range), mse.ctypes.data, ms.ctypes.data if msssim else None,
                                                     self._stream()))
        return dict(mse=mse, psnr=-10.0 * np.log10(mse), msssim=ms)

    # ---- instrumentation ----------------------------------------------------------------------------
    def saturation_count(self, reset: bool = True) -> int:
        """Elements of the fp16 operand planes clipped at +-65504 since the last reset (needs set_option("check_saturation", 1));
        synchronises the current stream."""
        n = ctypes.c_int64()
        with torch.cuda.device(self._device):
            _lib.check(_lib.lib().lbic_saturation_count(self._need(), self._stream(), ctypes.byref(n), 1 if reset else 0))
        return int(n.value)

    def launch_count(self) -> int:
        return int(_lib.lib().lbic_launch_count(self._need()))

    def set_profiling(self, on: bool):
        _lib.check(_lib.lib().lbic_set_profiling(self._need(), 1 if on else 0))

    def get_profile(self):
        n, ms, fl = ctypes.c_int64(), ctypes.c_double(), ctypes.c_double()
        _lib.check(_lib.lib().lbic_get_profile(self._need(), ctypes.byref(n), ctypes.byref(ms), ctypes.byref(fl)))
        return dict(gemm_launches=n.value, gemm_ms=ms.value, gemm_flops=fl.value)

    LAYER_NAMES = ("E0", "E1", "E2", "E3", "F0", "G0", "F1", "G1", "F2", "G2", "F3",
                   "D0", "IG0", "D1", "IG1", "D2", "IG2", "D3")

    def get_layer_profile(self):
        """Per-layer launch count, device ms and algorithmic FLOPs of the GEMM launches recorded since
        set_profiling(True)."""
        n = len(self.LAYER_NAMES)
        cnt, ms, fl = (ctypes.c_int64 * n)(), (ctypes.c_double * n)(), (ctypes.c_double * n)()
        got = _lib.lib().lbic_get_layer_profile(self._need(), n, cnt, ms, fl)
        if got < 0:
            _lib.check(got)
        return {self.LAYER_NAMES[i]: dict(launches=cnt[i], ms=ms[i], flops=fl[i]) for i in range(got)}

    def debug_gemm(self, A, W):
        """D = A @ W.T through the selected GEMM core (bring-up/test hook)."""
        A, W = A.contiguous().float(), W.contiguous().float()
        D = torch.empty(A.shape[0], W.shape[0], device=A.device, dtype=torch.float32)
        with torch.cuda.device(A.device):
            _lib.check(_lib.lib().lbic_debug_gemm(self._need(), A.data_ptr(), W.data_ptr(), D.data_ptr(), A.shape[0],
                                                  A.shape[1], W.shape[0], self._stream()))
        return D

    EPI_MODES = ("lrelu", "pregdn", "gdn", "igdn", "ksi", "quant", "recon", "raw", "resid")   # lbic_debug_layer_args.mode
    DEBUG_CORES = ("simt", "tc", "ws", "pair", "pair_wide")                                   # lbic_debug_layer_args.core

    def debug_layer(self, mode, A, W, core="tc", force_bn=0, bias=None, aux=None, acc_scale=1.0, M=None,
                    scale_table=None, no_clamp=False):
        """ONE fused GEMM layer (test hook, lbic_debug_layer): A / W are lists of one or two fp32 CUDA tensors (R, K_s) /
        (cout, K_s); aux (R, ld_aux) is the pre-GDN activation, ksi (scales | means) or the residual; scale_table (64,)
        CUDA fp32 or None for the installed table.  Returns the planes the mode writes: 'f32' (R, cout) fp32 (RAW, PREGDN,
        KSI, RECON, RESID), 'sym' (R, M) int32 and 'idx' (R, M) uint8 (QUANT), 'hi' / 'lo' (R, cout) fp16."""
        md = self.EPI_MODES.index(mode)
        A = [a.contiguous().float() for a in A]
        W = [w.contiguous().float() for w in W]
        R, cout, dev = A[0].shape[0], W[0].shape[0], A[0].device
        M = cout if M is None else int(M)
        keep = list(A) + list(W)
        a = _lib.LbicDebugLayerArgs()
        a.mode, a.core, a.force_bn, a.R, a.cout, a.nseg = md, self.DEBUG_CORES.index(core), int(force_bn), R, cout, len(A)
        for s in range(len(A)):
            a.K[s], a.A[s], a.W[s] = A[s].shape[1], A[s].data_ptr(), W[s].data_ptr()
        if bias is not None:
            bias = bias.contiguous().float()
            keep.append(bias)
            a.bias = bias.data_ptr()
        if aux is not None:
            aux = aux.contiguous().float()
            keep.append(aux)
            a.aux, a.ld_aux = aux.data_ptr(), aux.shape[1]
        if scale_table is not None:
            scale_table = scale_table.contiguous().float().to(dev)
            keep.append(scale_table)
            a.scale_table = scale_table.data_ptr()
        a.acc_scale, a.M, a.no_clamp = float(acc_scale), M, 1 if no_clamp else 0
        out = {}
        if mode == "quant":
            out["sym"] = torch.empty(R, M, dtype=torch.int32, device=dev)
            out["idx"] = torch.empty(R, M, dtype=torch.uint8, device=dev)
            a.out_f32, a.out_idx = out["sym"].data_ptr(), out["idx"].data_ptr()
        elif mode in ("raw", "pregdn", "ksi", "recon", "resid"):
            out["f32"] = torch.empty(R, cout, dtype=torch.float32, device=dev)
            a.out_f32 = out["f32"].data_ptr()
        if mode in ("lrelu", "pregdn", "gdn", "igdn", "quant"):
            out["hi"] = torch.empty(R, cout, dtype=torch.float16, device=dev)
            out["lo"] = torch.empty(R, cout, dtype=torch.float16, device=dev)
            a.out_hi, a.out_lo = out["hi"].data_ptr(), out["lo"].data_ptr()
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().lbic_debug_layer(self._need(), ctypes.byref(a), self._stream()))
        del keep
        return out

    def debug_selfinfo(self, ksi, sym):
        """-log2 likelihood of the symbols sym (R, M) int32 under the scales ksi[:, :M] (test hook, lbic_debug_selfinfo)."""
        ksi, sym = ksi.contiguous().float(), sym.contiguous().int()
        R, M = sym.shape
        info = torch.empty(R, M, dtype=torch.float32, device=sym.device)
        with torch.cuda.device(sym.device):
            _lib.check(_lib.lib().lbic_debug_selfinfo(self._need(), ksi.data_ptr(), ksi.shape[1], sym.data_ptr(), R, M,
                                                      info.data_ptr(), self._stream()))
        return info

    def debug_scale_index(self, scales, scale_table):
        """CDF indexes of fp32 CUDA scales by the decoders' bisection and by their hinted lookup (test hook,
        lbic_debug_scale_index) -> (idx_bisect, idx_hinted) int32."""
        scales, tab = scales.contiguous().float(), scale_table.contiguous().float().to(scales.device)
        ib, ih = (torch.empty(scales.numel(), dtype=torch.int32, device=scales.device) for _ in range(2))
        with torch.cuda.device(scales.device):
            _lib.check(_lib.lib().lbic_debug_scale_index(self._need(), scales.data_ptr(), scales.numel(), tab.data_ptr(),
                                                         ib.data_ptr(), ih.data_ptr(), self._stream()))
        return ib, ih

    def debug_rans_encode(self, sym, idx, seg, form, stream_cap):
        """The streams [seg[s], seg[s+1]) of sym (int32) / idx (uint8) CUDA tensors through rANS encoder form 1 (warp), 2
        (CTA) or 3 (thread per stream) (test hook, lbic_debug_rans_encode) -> list of stream bytes."""
        seg = torch.as_tensor(seg, dtype=torch.int64).to(sym.device)
        n = seg.numel() - 1
        if sym.numel() == 0:                 # streams of no symbols: any valid (non-null) arrays
            sym, idx = torch.zeros(4, dtype=torch.int32, device=sym.device), torch.zeros(4, dtype=torch.uint8, device=sym.device)
        out = torch.zeros(n, stream_cap, dtype=torch.uint8, device=sym.device)
        lens = torch.zeros(n, dtype=torch.int32, device=sym.device)
        with torch.cuda.device(sym.device):
            _lib.check(_lib.lib().lbic_debug_rans_encode(self._need(), sym.data_ptr(), idx.data_ptr(), n, seg.data_ptr(),
                                                         int(form), out.data_ptr(), stream_cap, lens.data_ptr(),
                                                         self._stream()))
        out_h, lens_h = out.cpu().numpy(), lens.cpu().numpy()
        return [out_h[s, :lens_h[s]].tobytes() for s in range(n)]

    def debug_rans_decode_steps(self, streams, ksi, M, n_steps, form):
        """Reference-container streams (list of bytes) decoded in n_steps steps of M symbols with scales | means from ksi
        (n_steps * n_streams, 2M) CUDA fp32 through decode form 0 (whole stream), 1 (warp, int32 tables), 2 (warp,
        shared-memory tables) or 3 (thread per row) (test hook, lbic_debug_rans_decode_steps) -> (sym (n_steps, n_streams,
        M) int32, yq_hi, yq_lo fp16 of that shape, words consumed per stream); form 0 returns symbols only."""
        n, dev = len(streams), ksi.device
        cap = max(8, max(len(s) for s in streams) + 3) // 4 * 4
        buf = np.zeros((n, cap), dtype=np.uint8)
        for s, b in enumerate(streams):
            buf[s, :len(b)] = np.frombuffer(b, dtype=np.uint8)
        d_buf = torch.from_numpy(buf).to(dev)
        lens = torch.tensor([len(b) for b in streams], dtype=torch.int32, device=dev)
        ksi = ksi.contiguous().float()
        sym = torch.empty(n_steps, n, M, dtype=torch.int32, device=dev)
        hi, lo = (torch.empty(n_steps, n, M, dtype=torch.float16, device=dev) for _ in range(2))
        pos = torch.zeros(n, dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().lbic_debug_rans_decode_steps(self._need(), d_buf.data_ptr(), lens.data_ptr(), cap, n, M,
                                                               n_steps, ksi.data_ptr(), int(form), sym.data_ptr(),
                                                               hi.data_ptr(), lo.data_ptr(), pos.data_ptr(), self._stream()))
        return (sym, None, None, None) if form == 0 else (sym, hi, lo, pos)

    def debug_compact_tables(self):
        """The compact tables of the installed CDFs (test hook, lbic_debug_compact_tables) -> (total, rows uint16 [total],
        offsets int32 [65], lut uint16 [64, 257]); total 0 (and None for the arrays) when the tables are too large for them."""
        total = ctypes.c_int()
        h = self._need()
        _lib.check(_lib.lib().lbic_debug_compact_tables(h, ctypes.byref(total), None, None, None))
        if total.value == 0:
            return 0, None, None, None
        rows = np.empty(total.value, dtype=np.uint16)
        off = np.empty(65, dtype=np.int32)
        lut = np.empty((64, 257), dtype=np.uint16)
        _lib.check(_lib.lib().lbic_debug_compact_tables(h, None, rows.ctypes.data, off.ctypes.data, lut.ctypes.data))
        return total.value, rows, off, lut


class BlkBasedPostProcessing:
    """Mirror of the reference's optional post-processing module (graphs/models/BlockBasedImgCompLossy_net.py:455-476,
    `use_postpm`): `out = x + pad(conv1x1(lrelu(conv3x3_valid(x))))` on the (n, 3B^2, Hb, Wb) block tensor of a
    reconstruction, as eval_model applies it (AGENT:604-606).  Runs in liblbic_b200 on the device of the codec model it
    is bound to (it shares that model's workspace); `state_dict` keys are the reference module's: res_net.0.weight
    (4C, C, 3, 3), res_net.0.bias, res_net.2.weight (C, 4C, 1, 1), res_net.2.bias with C = 3B^2."""

    KEYS = ("res_net.0.weight", "res_net.0.bias", "res_net.2.weight", "res_net.2.bias")

    def __init__(self, model: BlockBasedImgCompLossyNetv9):
        self.model = model
        self._sd = None

    def eval(self):
        return self

    def to(self, device):
        return self

    def load_state_dict(self, state_dict, strict: bool = True):
        missing = [k for k in self.KEYS if k not in state_dict]
        if missing:
            raise RuntimeError(f"Missing key(s) in state_dict: {missing}")
        C = self.model.Cin
        want = {"res_net.0.weight": (4 * C, C, 3, 3), "res_net.0.bias": (4 * C,), "res_net.2.weight": (C, 4 * C, 1, 1),
                "res_net.2.bias": (C,)}
        keep, descs = [], []
        for k in self.KEYS:
            t = state_dict[k].detach().to(torch.float32).contiguous()
            if tuple(t.shape) != want[k]:
                raise RuntimeError(f"size mismatch for {k}: {tuple(t.shape)} vs {want[k]}")
            keep.append(t)
            d = _lib.LbicTensorDesc()
            d.name, d.data, d.ndim = k.encode(), t.data_ptr(), t.dim()
            for i, n in enumerate(t.shape):
                d.shape[i] = n
            descs.append(d)
        arr = (_lib.LbicTensorDesc * len(descs))(*descs)
        m = self.model
        with torch.cuda.device(m._device):
            _lib.check(_lib.lib().lbic_load_postpm_weights(m._need(), arr, len(descs), m._stream()))
        self._sd = OrderedDict((k, state_dict[k].detach().clone()) for k in self.KEYS)
        return SimpleNamespace(missing_keys=[], unexpected_keys=[])

    def state_dict(self):
        return OrderedDict(self._sd or {})

    def forward(self, x, clamp: bool = False):
        """x: (n, 3B^2, Hb, Wb) CUDA fp32 -> same shape; clamp=True folds in the caller's clamp_(-0.5, 0.5) (AGENT:606)."""
        m = self.model
        if not (x.is_cuda and x.dtype == torch.float32 and x.dim() == 4 and x.shape[1] == m.Cin):
            raise ValueError(f"x must be a CUDA fp32 tensor of shape (n, {m.Cin}, Hb, Wb)")
        x = x.contiguous()
        out = torch.empty_like(x)
        n, _, Hb, Wb = x.shape
        with torch.cuda.device(x.device):
            _lib.check(_lib.lib().lbic_postprocess(m._need(), x.data_ptr(), n, Hb, Wb, out.data_ptr(), 1 if clamp else 0,
                                                   m._stream()))
        return out

    __call__ = forward
