"""Host-side owner of a libgnnb context: uploads GNN parameters and the verified network once, then scores
frontiers of subdomains through the C ABI (include/gnnb.h).  PyTorch is used for device memory and streams only."""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Tuple

import torch

from . import _lib
from .frontier import Frontier
from .networks import NetSpec

# state_dict order of the 26 linears (graph_conv.py:36-74, 431-432) — the order gnnb_set_gnn_weights expects
UPDATE_LINEARS = ['inp_f', 'inp_f_1', 'inp_b', 'inp_b_1', 'inp_b2', 'inp_b2_2', 'fc1', 'fc1_1', 'fc3', 'fc3_2',
                  'fc4', 'fc4_2', 'out1', 'out2', 'out3', 'bc1', 'bc1_1', 'bc1_2', 'bc2', 'bc2_1', 'bc3', 'bc3_1',
                  'bc4', 'bc4_1']
SCORE_LINEARS = ['fnode', 'fscore']
STATE_DICT_KEYS = ([f'EmbedUpdates.update.{n}.{s}' for n in UPDATE_LINEARS for s in ('weight', 'bias')]
                   + [f'ComputeFinalScore.{n}.{s}' for n in SCORE_LINEARS for s in ('weight', 'bias')])

_MATH = {'tc': _lib.MATH_TC_FP16X3, 'simt': _lib.MATH_SIMT_FP32}
# nn.Linear shapes of the 26 linears, same order (graph_conv.py:36-74, 431-432)
_LIN_IN = [3, 64, 2, 64, 128, 64, 7, 64, 128, 64, 128, 64, 4, 128, 64, 7, 64, 64, 192, 64, 128, 64, 128, 64, 64, 64]
_LIN_OUT = [64] * 25 + [1]


class Scorer:
    """One libgnnb context bound to one CUDA device.

    ``rescore``: in tensor-core mode, score the subdomains whose activations left the fp16 operand range (a NaN in an
    embedding) again in exact fp32 on the same GPU instead of failing the call (option "rescore" of include/gnnb.h)."""

    def __init__(self, device: int = 0, math: Optional[str] = None, chunk: int = 0, rescore: bool = False):
        if not torch.cuda.is_available():
            raise RuntimeError('gnn_branching_b200 needs a CUDA device (sm_100a); there is no CPU path')
        self.lib = _lib.load()
        self.device = int(device)
        h = C.c_void_p()
        st = self.lib.gnnb_create(C.byref(h), self.device)
        if st != _lib.GNNB_OK:
            raise _lib.GnnbError(st, 'gnnb_create failed (see stderr)')
        self.h = h
        self._net_key = None
        self._gnn_key = None
        self.net: Optional[NetSpec] = None
        if math is not None:
            self.set_option('math', _MATH[math])
        if chunk:
            self.set_option('chunk', chunk)
        if rescore:
            self.set_option('rescore', 1)

    def __del__(self):
        h, self.h = getattr(self, 'h', None), None
        if h:
            try:
                self.lib.gnnb_destroy(h)
            except Exception:
                pass

    # ---- helpers ----
    def _raise(self, st: int):
        buf = C.create_string_buffer(512)
        self.lib.gnnb_last_error(self.h, buf, 512)
        raise _lib.GnnbError(st, buf.value.decode(errors='replace'))

    def _ok(self, st: int):
        if st != _lib.GNNB_OK:
            self._raise(st)

    def set_option(self, key: str, value: int):
        self._ok(self.lib.gnnb_set_option(self.h, key.encode(), int(value)))

    def get_option(self, key: str) -> int:
        return int(self.lib.gnnb_get_option(self.h, key.encode()))

    @property
    def launches(self) -> int:
        return int(self.lib.gnnb_launch_count(self.h))

    @property
    def rescored(self) -> int:
        """Subdomains the last scoring call scored again in exact fp32 (option ``rescore``)."""
        return self.get_option('rescored')

    # ---- parameters ----
    def set_gnn(self, state_dict: Dict[str, torch.Tensor], T: int = 2, p: int = 64, key=None, force: bool = False):
        """Upload the 52 GNN tensors (models/cifar_trained_gnn/*.pt loads unchanged).

        Caching contract: with a ``key`` the upload is skipped when the key equals the one of the last upload.  Callers
        derive keys from (data_ptr, _version) of the tensors, which does NOT see writes that bypass the version counter
        (``p.data.copy_()``, writes through a numpy view, some custom optimizers): after such writes pass ``force=True``
        (or call ``invalidate()``)."""
        if not force and key is not None and key == self._gnn_key:
            return
        missing = [k for k in STATE_DICT_KEYS if k not in state_dict]
        if missing:
            raise KeyError(f'state_dict is missing {missing[:3]}...')
        host = [state_dict[k].detach().to('cpu', torch.float32).contiguous() for k in STATE_DICT_KEYS]
        ptrs, keep = _lib.fptr_array(host)
        numels = (C.c_int64 * len(host))(*[t.numel() for t in host])
        self._ok(self.lib.gnnb_set_gnn_weights(self.h, ptrs, numels, len(host), int(T), int(p)))
        self._gnn_key = key
        del keep

    def invalidate(self):
        """Forget the cache keys: the next set_gnn / set_network uploads again whatever its key."""
        self._gnn_key = None
        self._net_key = None

    def set_network(self, net: NetSpec, key=None, force: bool = False):
        """Upload the verified network (same caching contract as ``set_gnn``)."""
        if not force and key is not None and key == self._net_key:
            return
        descs = (_lib.LayerDesc * net.L)()
        keep = []
        for k, a in enumerate(net.affine):
            w = a.weight.detach().to('cpu', torch.float32).contiguous()
            b = a.bias.detach().to('cpu', torch.float32).contiguous()
            keep += [w, b]
            d = descs[k]
            if a.kind == 'conv':
                d.kind = _lib.LAYER_CONV
                d.c_in, d.h_in, d.w_in = a.in_shape
                d.c_out, d.h_out, d.w_out = a.out_shape
                d.ksize, d.stride, d.pad = int(a.weight.shape[2]), int(a.stride), int(a.padding)
            else:
                d.kind = _lib.LAYER_LINEAR
                d.c_in, d.h_in, d.w_in = a.n_in, 1, 1
                d.c_out, d.h_out, d.w_out = a.n_out, 1, 1
                d.ksize, d.stride, d.pad = 1, 1, 0
            d.weight, d.bias = _lib.fptr(w), _lib.fptr(b)
        c0, h0, w0 = net.input_shape
        self._ok(self.lib.gnnb_set_network(self.h, descs, net.L, c0, h0, w0))
        self.net = net
        self._net_key = key
        del keep

    # ---- scoring ----
    def score(self, fr: Frontier, return_scores: bool = True, check: bool = True
              ) -> Tuple[torch.Tensor, torch.Tensor, Optional[torch.Tensor]]:
        """Score every subdomain of ``fr``.

        ``fr`` on the CUDA device: zero-copy, results are CUDA tensors.  ``fr`` on the CPU: inputs are copied
        host->device and results device->host inside the call (pin the frontier for full copy speed).
        Returns (best_score [B] f32, best_idx [B] i32, scores [B, sum n_k] f32 or None).
        """
        return self._score(fr, None, return_scores, check)

    def score_topk(self, fr: Frontier, k: int, return_scores: bool = False, check: bool = True
                   ) -> Tuple[torch.Tensor, torch.Tensor, Optional[torch.Tensor]]:
        """Score every subdomain of ``fr`` and return its ``k`` best branching candidates (1 <= k <= 64), device and host
        frontiers as in ``score``.  Returns (top_score [B, k] f32, top_idx [B, k] i32, scores [B, sum n_k] f32 or None).
        Order: NaN scores first, then descending score, ties by ascending flat index; (-inf, -1) past the last candidate.
        Column 0 is ``score``'s (best_score, best_idx) bit for bit."""
        if not 1 <= int(k) <= _lib.TOPK_MAX:
            raise ValueError(f'k must be in [1, {_lib.TOPK_MAX}], got {k}')
        return self._score(fr, int(k), return_scores, check)

    def topk(self, scores: torch.Tensor, k: int, mask: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
        """The ``k`` best entries of every row of ``scores`` [B, n] (CUDA) among those with ``mask`` != 0 (``mask`` [B, n] or
        None = every entry), in ``score_topk``'s order: (top_score [B, k] f32, top_idx [B, k] i32), CUDA tensors."""
        if not 1 <= int(k) <= _lib.TOPK_MAX:
            raise ValueError(f'k must be in [1, {_lib.TOPK_MAX}], got {k}')
        if not scores.is_cuda or scores.dim() != 2:
            raise ValueError('scores must be a [B, n] CUDA tensor')
        B, n = int(scores.shape[0]), int(scores.shape[1])
        scores = self._as_f32(scores, (B, n))
        if mask is not None:
            if not mask.is_cuda:
                raise ValueError('mask must be a CUDA tensor')
            mask = self._as_f32(mask, (B, n))
        top_score = torch.empty(B, int(k), dtype=torch.float32, device=scores.device)
        top_idx = torch.empty(B, int(k), dtype=torch.int32, device=scores.device)
        if B == 0:
            return top_score, top_idx
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            self._ok(self.lib.gnnb_topk(self.h, B, n, _lib.fptr(scores), _lib.fptr(mask) if mask is not None else None, int(k),
                                        _lib.fptr(top_score), C.cast(top_idx.data_ptr(), C.POINTER(C.c_int32)), C.c_void_p(stream)))
        return top_score, top_idx

    def _frontier_desc(self, fr: Frontier):
        """gnnb_frontier of every array of ``fr`` (on this scorer's GPU, or on the CPU) + the objects that keep its arrays
        alive."""
        if self.net is None:
            raise RuntimeError('set_network first')
        net, B, L = self.net, fr.B, self.net.L
        host = fr.device.type == 'cpu'
        if not host and fr.device.index not in (None, self.device):
            raise ValueError(f'frontier is on {fr.device}, scorer on cuda:{self.device}')
        sizes = [net.n0] + net.hidden_sizes + [1]

        def f(t, shape):
            if t.device != fr.device:
                raise ValueError(f'frontier tensors live on different devices ({t.device} vs {fr.device})')
            return self._as_f32(t, shape)

        lb = [f(fr.lb[k], (B, sizes[k])) for k in range(L + 2)]
        ub = [f(fr.ub[k], (B, sizes[k])) for k in range(L + 2)]
        dual = [f(fr.dual[k], (B, sizes[k + 1], 3)) for k in range(L)]
        pre = [f(fr.prim_pre[k], (B, sizes[k + 1])) for k in range(L)]
        post = [f(fr.prim_post[k], (B, sizes[k + 1])) for k in range(L)]
        flat = [f(fr.prim_out, (B,)), f(fr.primal_input, (B, net.n0)), f(fr.Wp, (B, sizes[L])), f(fr.bp, (B,)),
                f(fr.mask, (B, net.n_hidden))]
        d = _lib.FrontierDesc()
        d.B, d.mem = B, (_lib.MEM_HOST if host else _lib.MEM_DEVICE)
        keep = [lb, ub, dual, pre, post, flat]
        for name, arrs in (('lb', lb), ('ub', ub), ('dual', dual), ('prim_pre', pre), ('prim_post', post)):
            p, k = _lib.fptr_array(arrs)
            setattr(d, name, p)
            keep.append(k)
        d.prim_out, d.primal_input, d.wp, d.bp, d.mask = map(_lib.fptr, flat)
        return d, keep

    def _score(self, fr: Frontier, n_top: Optional[int], return_scores: bool, check: bool):
        """gnnb_score (n_top = None) or gnnb_score_topk with k = n_top."""
        d, keep = self._frontier_desc(fr)
        B, dev = fr.B, fr.device
        host = dev.type == 'cpu'
        pinned = host and torch.cuda.is_available()      # pinned results: device->host copies stay asynchronous
        shape = (B,) if n_top is None else (B, n_top)
        best = torch.empty(shape, dtype=torch.float32, device=dev, pin_memory=pinned)
        idx = torch.empty(shape, dtype=torch.int32, device=dev, pin_memory=pinned)
        scores = torch.empty(B, self.net.n_hidden, dtype=torch.float32, device=dev, pin_memory=pinned) if return_scores else None
        if B == 0:
            return best, idx, scores
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            out = (_lib.fptr(best), C.cast(idx.data_ptr(), C.POINTER(C.c_int32)), _lib.fptr(scores) if scores is not None else None,
                   C.c_void_p(stream))
            if n_top is None:
                st = self.lib.gnnb_score(self.h, C.byref(d), *out)
            else:
                st = self.lib.gnnb_score_topk(self.h, C.byref(d), n_top, *out)
            if st != _lib.GNNB_OK:
                self._raise(st)
            if check and not host:
                self.check()
        del keep
        return best, idx, scores

    def score_winners(self, fr: Frontier, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Score every subdomain of ``fr`` (CUDA or pinned CPU) and return the winners as packed records on the GPU:
        int32 ``[B, 2]`` = (bit pattern of the fp32 score, flat index) — the buffer the multi-GPU winner all-gather sends
        (``dist.gather_winner_records``); ``out``: a preallocated ``[>= B, 2]`` int32 CUDA tensor to write into."""
        d, keep = self._frontier_desc(fr)
        dev = torch.device('cuda', self.device)
        if out is None:
            out = torch.empty(fr.B, 2, dtype=torch.int32, device=dev)
        if out.dtype != torch.int32 or not out.is_cuda or not out.is_contiguous() or out.shape[0] < fr.B or out.shape[1:] != (2,):
            raise ValueError('out must be a contiguous int32 CUDA tensor [>= B, 2]')
        if fr.B:
            with torch.cuda.device(self.device):
                stream = torch.cuda.current_stream().cuda_stream
                self._ok(self.lib.gnnb_score_winners(self.h, C.byref(d), C.c_void_p(out.data_ptr()), None, C.c_void_p(stream)))
        del keep
        return out[:fr.B]

    def babsr(self, fr: Frontier, icp_score_counter=None, random_order=None, sparsest_layer: int = 0,
              decision_threshold: float = 0.001, return_scores: bool = False):
        """BaBSR / KW heuristic decisions for every subdomain of ``fr`` (plnn/kw_score_conv.py:41-156, batched).

        Returns (decision [B, 2] i32 = (layer, index in layer), counters [B] i32, kind [B] i32, scores or None);
        tensors live where ``fr`` lives."""
        if self.net is None:
            raise RuntimeError('set_network first')
        net, B = self.net, fr.B
        L = net.L
        host = fr.device.type == 'cpu'
        sizes = [net.n0] + net.hidden_sizes + [1]
        lb = [self._as_f32(fr.lb[k], (B, sizes[k])) for k in range(L + 2)]
        ub = [self._as_f32(fr.ub[k], (B, sizes[k])) for k in range(L + 2)]
        wp, mask = self._as_f32(fr.Wp, (B, sizes[L])), self._as_f32(fr.mask, (B, net.n_hidden))
        dev = fr.device
        if random_order is None:                                  # relu_conv_gnnkwthreshold.py:98-101
            random_order = [sparsest_layer] + [k for k in range(L) if k != sparsest_layer] if sparsest_layer >= 0 else list(range(L))
        random_order = [int(k) for k in random_order]
        if sorted(random_order) != list(range(L)):                # a short list would be zero-padded silently, a long one overflow
            raise ValueError(f'random_order must be a permutation of range({L}), got {random_order}')
        order = (C.c_int32 * L)(*random_order)
        cin = None
        if icp_score_counter is not None:
            cin = torch.as_tensor(icp_score_counter, dtype=torch.int32).to(dev).contiguous()
        dec = torch.empty(B, 2, dtype=torch.int32, device=dev)
        cout = torch.empty(B, dtype=torch.int32, device=dev)
        kind = torch.empty(B, dtype=torch.int32, device=dev)
        scores = torch.empty(B, net.n_hidden, dtype=torch.float32, device=dev) if return_scores else None
        if B == 0:
            return dec, cout, kind, scores
        d = _lib.FrontierDesc()
        d.B, d.mem = B, (_lib.MEM_HOST if host else _lib.MEM_DEVICE)
        plb, k1 = _lib.fptr_array(lb)
        pub, k2 = _lib.fptr_array(ub)
        d.lb, d.ub, d.wp, d.mask = plb, pub, _lib.fptr(wp), _lib.fptr(mask)
        ip = lambda t: C.cast(t.data_ptr(), C.POINTER(C.c_int32)) if t is not None else None
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            self._ok(self.lib.gnnb_babsr(self.h, C.byref(d), int(sparsest_layer), float(decision_threshold), order, ip(cin),
                                         ip(dec), ip(cout), ip(kind), _lib.fptr(scores) if scores is not None else None,
                                         C.c_void_p(stream)))
        del k1, k2
        return dec, cout, kind, scores

    # ---- online fine-tuning (graph_score_online.py:62-77) ----
    def score_grad(self, fr: Frontier, terms) -> torch.Tensor:
        """Back-propagate ``sum_i coeff_i * score[domain_i][flat_index_i]`` into the gradient buffers of the context
        (zeroed first, like ``optimizer.zero_grad(); loss.backward()``).  ``terms``: iterable of (domain, flat index,
        coeff); returns the terms' scores (fp32, CPU).  Or ``terms`` = (domain int32, index int32, coeff float32), three
        CUDA tensors [n] on this scorer's GPU (``gnnb_score_grad_device``): a term with domain < 0 is inactive, one out of
        range is skipped and counted (option ``grad_bad_terms``), both score NaN; returns the scores as a CUDA tensor [n],
        and nothing but the count of named subdomains is read back."""
        if isinstance(terms, tuple) and len(terms) == 3 and all(isinstance(t, torch.Tensor) for t in terms):
            return self._score_grad_device(fr, *terms)
        terms = list(terms)
        nt = len(terms)
        dom = (C.c_int32 * nt)(*[int(t[0]) for t in terms])
        idx = (C.c_int32 * nt)(*[int(t[1]) for t in terms])
        coeff = (C.c_float * nt)(*[float(t[2]) for t in terms])
        out = (C.c_float * nt)()
        d, keep = self._frontier_desc(fr)
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            self._ok(self.lib.gnnb_score_grad(self.h, C.byref(d), nt, dom, idx, coeff, out, C.c_void_p(stream)))
        del keep
        return torch.tensor(list(out), dtype=torch.float32)

    def _score_grad_device(self, fr: Frontier, dom: torch.Tensor, idx: torch.Tensor, coeff: torch.Tensor) -> torch.Tensor:
        dev = torch.device('cuda', self.device)
        n = int(dom.numel())
        for t, dt in ((dom, torch.int32), (idx, torch.int32), (coeff, torch.float32)):
            if t.device != dev or t.dtype != dt or t.dim() != 1 or t.numel() != n:
                raise ValueError(f'device terms must be [n] tensors on {dev}: domain / index int32, coeff float32')
        dom, idx, coeff = dom.contiguous(), idx.contiguous(), coeff.contiguous()
        out = torch.empty(n, dtype=torch.float32, device=dev)
        d, keep = self._frontier_desc(fr)
        ip = lambda t: C.cast(t.data_ptr(), C.POINTER(C.c_int32))
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            self._ok(self.lib.gnnb_score_grad_device(self.h, C.byref(d), n, ip(dom), ip(idx), _lib.fptr(coeff), _lib.fptr(out),
                                                     C.c_void_p(stream)))
        del keep
        return out

    def copy_weights_to(self, tensors) -> None:
        """Copy the parameters the context scores with into 52 contiguous fp32 tensors in state_dict order, on the CPU or on
        this scorer's GPU (device to device, no host round trip)."""
        tensors = list(tensors)
        for t in tensors:
            if t.dtype != torch.float32 or not t.is_contiguous() or (t.is_cuda and t.device.index != self.device):
                raise ValueError('copy_weights_to needs contiguous fp32 tensors on the CPU or on the scorer\'s GPU')
        ptrs, keep = _lib.fptr_array(tensors)
        numels = (C.c_int64 * len(tensors))(*[t.numel() for t in tensors])
        self._ok(self.lib.gnnb_get_gnn_weights(self.h, ptrs, numels, len(tensors)))
        del keep

    def _download(self, fn) -> Dict[str, torch.Tensor]:
        shapes = []
        for l in range(len(_LIN_IN)):
            shapes += [(_LIN_OUT[l], _LIN_IN[l]), (_LIN_OUT[l],)]
        host = [torch.empty(s, dtype=torch.float32) for s in shapes]
        ptrs, keep = _lib.fptr_array(host)
        numels = (C.c_int64 * len(host))(*[t.numel() for t in host])
        self._ok(fn(self.h, ptrs, numels, len(host)))
        del keep
        return dict(zip(STATE_DICT_KEYS, host))

    def gradients(self) -> Dict[str, torch.Tensor]:
        """The reference's ``p.grad`` after ``loss.backward()``, keyed like the state_dict (CPU tensors)."""
        return self._download(self.lib.gnnb_get_gradients)

    def weights(self) -> Dict[str, torch.Tensor]:
        """The parameters the context currently scores with (the reference's ``model.state_dict()``)."""
        return self._download(self.lib.gnnb_get_gnn_weights)

    def adam_step(self, lr: float, weight_decay: float = 0.0, betas=(0.9, 0.999), eps: float = 1e-8):
        """One ``torch.optim.Adam`` step on the device with the gradients of the last ``score_grad``."""
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            self._ok(self.lib.gnnb_adam_step(self.h, float(lr), float(betas[0]), float(betas[1]), float(eps),
                                             float(weight_decay), C.c_void_p(stream)))
        self._gnn_key = None

    def adam_reset(self):
        self._ok(self.lib.gnnb_adam_reset(self.h))

    # ---- batched KW bounds (gnnb_kw.cu) ----
    def _kw_io(self, x: torch.Tensor, Wp: torch.Tensor, bp: torch.Tensor, with_mask: bool):
        """Inputs and outputs of the KW bound entries: B, the layer sizes, ``x`` [B, n0] (or [n0], shared), ``Wp`` [B, n_L] and
        ``bp`` [B] as contiguous fp32 on this scorer's GPU, L + 2 output tensors [B, n_k] each for the lower and the upper
        bounds, and L int8 output masks with their pointer array (both None without ``with_mask``)."""
        if self.net is None:
            raise RuntimeError('set_network first')
        net, L = self.net, self.net.L
        dev = torch.device('cuda', self.device)
        sizes = [net.n0] + net.hidden_sizes + [1]
        Wp = Wp.to(dev, torch.float32).reshape(-1, sizes[L]).contiguous()
        B = int(Wp.shape[0])
        x = x.to(dev, torch.float32).reshape(-1, net.n0)
        x = (x.expand(B, net.n0) if x.shape[0] == 1 else x).contiguous()
        bp = bp.to(dev, torch.float32).reshape(B).contiguous()
        lbs = [torch.empty(B, n, dtype=torch.float32, device=dev) for n in sizes]
        ubs = [torch.empty(B, n, dtype=torch.float32, device=dev) for n in sizes]
        masks = mptr = None
        if with_mask:
            masks = [torch.empty(B, n, dtype=torch.int8, device=dev) for n in sizes[1:L + 1]]
            marr = (C.POINTER(C.c_int8) * L)(*[C.cast(m.data_ptr(), C.POINTER(C.c_int8)) for m in masks])
            mptr = C.cast(marr, C.POINTER(C.POINTER(C.c_int8)))      # keeps marr alive
        return B, sizes, x, Wp, bp, lbs, ubs, masks, mptr

    def kw_bounds(self, x: torch.Tensor, eps: float, Wp: torch.Tensor, bp: torch.Tensor, provided_lb=None, provided_ub=None):
        """KW intermediate bounds of B domains (init_kw_bounds of the reference, batched).  ``x`` [B, n0] (or [n0], shared),
        ``Wp`` [B, n_L], ``bp`` [B]; ``provided_lb`` / ``provided_ub``: L tensors [B, n_k] (the parent's pre-ReLU bounds with
        the split applied) or None.  Returns (lbs, ubs): L + 2 CUDA tensors [B, n_k] each."""
        B, sizes, x, Wp, bp, lbs, ubs, _, _ = self._kw_io(x, Wp, bp, with_mask=False)
        dev = x.device
        plb = pub = None
        keep = []
        if provided_lb is not None:
            pl = [self._as_f32(t.to(dev), (B, sizes[k + 1])) for k, t in enumerate(provided_lb)]
            pu = [self._as_f32(t.to(dev), (B, sizes[k + 1])) for k, t in enumerate(provided_ub)]
            plb, k1 = _lib.fptr_array(pl)
            pub, k2 = _lib.fptr_array(pu)
            keep += [pl, pu, k1, k2]
        olb, k3 = _lib.fptr_array(lbs)
        oub, k4 = _lib.fptr_array(ubs)
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            self._ok(self.lib.gnnb_kw_bounds(self.h, B, _lib.fptr(x), float(eps), _lib.fptr(Wp), _lib.fptr(bp), plb, pub, olb, oub,
                                             C.c_void_p(stream)))
            torch.cuda.synchronize()
        del keep, k3, k4
        return lbs, ubs

    def root_bounds(self, x: torch.Tensor, eps: float, Wp: torch.Tensor, bp: torch.Tensor, with_mask: bool = True):
        """Bounds of B root domains — the bounds part of ``KWConvGen.build_the_model`` (plnn/conv_kwinter_gen.py:199-270):
        KW bounds intersected with interval bounds, and a KW pass where that moved a hidden layer.  ``x`` [B, n0] (or [n0]),
        ``Wp`` [B, n_L], ``bp`` [B].  Returns (lbs, ubs, masks, second_pass) like ``child_bounds``."""
        B, _, x, Wp, bp, lbs, ubs, masks, mptr = self._kw_io(x, Wp, bp, with_mask)
        second = torch.empty(B, dtype=torch.int32, device=x.device)
        olb, k3 = _lib.fptr_array(lbs)
        oub, k4 = _lib.fptr_array(ubs)
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            self._ok(self.lib.gnnb_root_bounds(self.h, B, _lib.fptr(x), float(eps), _lib.fptr(Wp), _lib.fptr(bp), olb, oub, mptr,
                                               C.cast(second.data_ptr(), C.POINTER(C.c_int32)), C.c_void_p(stream)))
        del k3, k4
        return lbs, ubs, masks, second

    def child_bounds(self, x: torch.Tensor, eps: float, Wp: torch.Tensor, bp: torch.Tensor, parent_lb, parent_ub,
                     dec_layer: torch.Tensor, dec_index: torch.Tensor, choice: torch.Tensor, with_mask: bool = True):
        """Bounds of B child domains — the bounds part of ``KWConvGen.update_the_model`` (plnn/conv_kwinter_gen.py:558-660),
        batched and device-resident.  ``parent_lb`` / ``parent_ub``: L + 2 tensors [B, n_k] (input box, pre-ReLU bounds,
        property output); ``dec_layer`` (0-based hidden layer), ``dec_index``, ``choice`` (0 blocked / 1 passing): [B] ints.
        Returns (lbs, ubs, masks, second_pass): L + 2 CUDA tensors [B, n_k] each, L int8 masks in the BaB convention
        (or None), [B] int32 flags of the domains that took the second KW pass."""
        B, sizes, x, Wp, bp, lbs, ubs, masks, mptr = self._kw_io(x, Wp, bp, with_mask)
        dev = x.device
        pl = [self._as_f32(t.to(dev).reshape(B, -1), (B, sizes[k])) for k, t in enumerate(parent_lb)]
        pu = [self._as_f32(t.to(dev).reshape(B, -1), (B, sizes[k])) for k, t in enumerate(parent_ub)]
        ints = [t.to(dev, torch.int32).reshape(B).contiguous() for t in (dec_layer, dec_index, choice)]
        second = torch.empty(B, dtype=torch.int32, device=dev)
        plb, k1 = _lib.fptr_array(pl)
        pub, k2 = _lib.fptr_array(pu)
        olb, k3 = _lib.fptr_array(lbs)
        oub, k4 = _lib.fptr_array(ubs)
        ip = lambda t: C.cast(t.data_ptr(), C.POINTER(C.c_int32))
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            self._ok(self.lib.gnnb_child_bounds(self.h, B, _lib.fptr(x), float(eps), _lib.fptr(Wp), _lib.fptr(bp), plb, pub,
                                                ip(ints[0]), ip(ints[1]), ip(ints[2]), olb, oub, mptr, ip(second), C.c_void_p(stream)))
        del k1, k2, k3, k4
        return lbs, ubs, masks, second

    def check(self) -> None:
        """Synchronise and raise if a NaN appeared in an embedding (the reference drops into pdb there)."""
        n = C.c_int64(0)
        with torch.cuda.device(self.device):
            st = self.lib.gnnb_check(self.h, C.c_void_p(torch.cuda.current_stream().cuda_stream), C.byref(n))
        if st != _lib.GNNB_OK:
            self._raise(st)

    def profile_reset(self):
        self._ok(self.lib.gnnb_profile_reset(self.h))

    def profile_read(self) -> Dict[str, dict]:
        """{kernel class: {'ms', 'launches', 'rows'}} accumulated while option 'profile' = 1."""
        out = {}
        for i, name in enumerate(_lib.KERNEL_CLASSES):
            ms, n, rows = C.c_double(0), C.c_int64(0), C.c_int64(0)
            self._ok(self.lib.gnnb_profile_read(self.h, i, C.byref(ms), C.byref(n), C.byref(rows)))
            out[name] = dict(ms=ms.value, launches=n.value, rows=rows.value)
        return out

    def snapshot(self, name: str) -> torch.Tensor:
        n = C.c_int64(0)
        self._ok(self.lib.gnnb_debug_snapshot(self.h, name.encode(), None, 0, C.byref(n)))
        out = torch.empty(n.value, dtype=torch.float32)
        self._ok(self.lib.gnnb_debug_snapshot(self.h, name.encode(), _lib.fptr(out), n.value, C.byref(n)))
        return out

    @staticmethod
    def _as_f32(t: torch.Tensor, shape) -> torch.Tensor:
        if tuple(t.shape) != tuple(shape):
            raise ValueError(f'expected shape {tuple(shape)}, got {tuple(t.shape)}')
        if t.dtype != torch.float32 or not t.is_contiguous():
            t = t.float().contiguous()
        return t


def flat_to_layer_index(flat_idx: int, hidden_sizes) -> list:
    """graph_score.py:43-47: flat ReLU index -> [dec_lay, dec_idx] via the cumulative layer sizes."""
    off = 0
    for lay, n in enumerate(hidden_sizes):
        if flat_idx < off + n:
            return [lay, flat_idx - off]
        off += n
    raise IndexError(flat_idx)
