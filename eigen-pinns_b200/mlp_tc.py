"""bf16 tensor-core back end of the corrector MLP ("perf mode"): host-side buffer management around
the tcgen05 kernels of csrc/mlp_tc.cu.  Same interface as engine.Fp32Mlp."""
import ctypes

import torch

from ._cabi import call, query, EpError


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def pack_rows(X, d_padded=None, out=None):
    """fp32 rows -> packed bf16 tiles [tile][d_p/8][128][8] (uint8 tensor)."""
    n, d = X.shape
    dp = d_padded if d_padded is not None else query("ep_tc_pad_features", d, 0)
    nbytes = query("ep_tc_packed_rows_bytes", n, dp)
    out = out if out is not None else torch.empty(nbytes, dtype=torch.uint8, device=X.device)
    call("ep_tc_pack_rows_bf16", n, d, dp, _p(X), X.stride(0), _p(out), _stream())
    return out


def unpack_rows(packed, n, d_padded):
    """Inverse of pack_rows for tests / debugging: (n, d_padded) fp32 tensor (torch ops, not a hot path)."""
    tiles = (n + 127) // 128
    t = packed.view(torch.bfloat16).view(tiles, d_padded // 8, 128, 8)
    return t.permute(0, 2, 1, 3).reshape(tiles * 128, d_padded)[:n].float()


def _table(values, ctype=ctypes.c_void_p):
    """Host array for the layer tables of ep_tc_chain_fwd_bf16 (device pointers or ints inside)."""
    arr = (ctype * len(values))()
    for i, v in enumerate(values):
        arr[i] = v if ctype is ctypes.c_int else (v.data_ptr() if v is not None else None)
    return arr


class TcMlp:
    """Forward: ONE launch for all layers (ep_tc_chain_fwd_bf16, CTA pairs).  chain_fwd=False runs the layer-by-layer
    kernels instead, the bit-exact reference the tests compare the chain against.  Backward, layer by layer from the
    top: the dW kernel of layer l (side stream) and the dX kernel that produces dZ of layer l - 1 (main stream) run
    concurrently on two disjoint shares of the SMs; layer 0 needs no dX, so its dW kernel takes the whole GPU."""

    def __init__(self, n, params, device, h=None, chain_fwd=True):
        self.p, self.n, self.dev = params, n, device
        self.chain_fwd = bool(chain_fwd)
        dims = params.dims                                    # [in, h1, ..., out]
        L = len(dims) - 1
        if L < 2:
            raise EpError("bf16 mode needs at least one hidden layer")
        self.L = L
        self.dims = dims
        self.pd = [query("ep_tc_pad_features", dims[0], 0)] + \
                  [query("ep_tc_pad_features", d, 1) for d in dims[1:-1]] + [query("ep_tc_pad_features", dims[-1], 0)]
        if max(self.pd) > 256:
            raise EpError("bf16 mode supports layer widths up to 256 (got %s)" % (dims,))
        u8 = dict(dtype=torch.uint8, device=device)
        rows = lambda d: torch.zeros(query("ep_tc_packed_rows_bytes", n, d), **u8)
        self.x0 = rows(self.pd[0])
        self.acts = [rows(self.pd[l + 1]) for l in range(L - 1)]             # outputs of hidden layers
        self.masks = [torch.zeros(query("ep_tc_relu_mask_bytes", n, self.pd[l + 1]), **u8) for l in range(L - 1)]
        wmax = max(self.pd[1:-1])
        self.dz = [rows(wmax) for _ in range(2)]
        self.dz_out = rows(self.pd[-1])
        self.Wp = [torch.zeros(query("ep_tc_packed_weight_bytes", self.pd[l + 1], self.pd[l]), **u8) for l in range(L)]
        self.WTp = [torch.zeros_like(w) for w in self.Wp]
        self.ws_bytes = query("ep_tc_dw_workspace_bytes")
        self.ws = torch.empty(self.ws_bytes, **u8)
        self.corr = torch.empty((n, dims[-1]), dtype=torch.float32, device=device)
        self.side_stream = torch.cuda.Stream(device=device)
        self.sm_count = torch.cuda.get_device_properties(device).multi_processor_count
        self.dx_share = 0.56           # measured: tools/dx_share_sweep.py, backward 2.11 -> 1.93 ms vs an even split
        self._packed_version = None
        self.want_corr = True          # engine sets False: only U_pred is needed inside the training step
        if self.chain_fwd:
            self._t_pd = _table(self.pd, ctypes.c_int)
            self._t_out = _table(dims[1:], ctypes.c_int)
            self._t_Wp, self._t_b = _table(self.Wp), _table(list(self.p.b))
            self._t_acts, self._t_masks = _table(self.acts), _table(self.masks)
        if h is not None:
            self.input_changed(h)

    def input_changed(self, h):
        pack_rows(h, self.pd[0], out=self.x0)
        self._packed_version = (h.data_ptr(), h._version)

    def _pack_weights(self):
        for l in range(self.L):
            W = self.p.W[l]
            call("ep_tc_pack_weight_bf16", W.shape[0], W.shape[1], self.pd[l + 1], self.pd[l], _p(W), _p(self.Wp[l]),
                 _p(self.WTp[l]) if l > 0 else None, _stream())

    def forward(self, h, U_base=None, scale=0.0, U_pred=None, scale_dev=None):
        if self._packed_version != (h.data_ptr(), h._version):
            self.input_changed(h)
        self._pack_weights()
        if self.chain_fwd:
            corr = self.corr if (self.want_corr or U_pred is None) else None
            call("ep_tc_chain_fwd_bf16", self.n, self.L, self._t_pd, self._t_out, _p(self.x0), self._t_Wp, self._t_b,
                 self._t_acts, self._t_masks, _p(corr), self.corr.stride(0), _p(U_base), float(scale), _p(scale_dev),
                 _p(U_pred), U_pred.stride(0) if U_pred is not None else 0, _stream())
            return self.corr
        x = self.x0
        for l in range(self.L - 1):
            call("ep_tc_linear_fwd_bf16", self.n, self.pd[l], self.dims[l + 1], self.pd[l + 1], _p(x), _p(self.Wp[l]),
                 _p(self.p.b[l]), 1, _p(self.acts[l]), _p(self.masks[l]), _stream())
            x = self.acts[l]
        l = self.L - 1
        call("ep_tc_linear_final_bf16", self.n, self.pd[l], self.dims[-1], self.pd[-1], _p(x), _p(self.Wp[l]),
             _p(self.p.b[l]), _p(self.corr), self.corr.stride(0), _p(U_base), float(scale), _p(scale_dev), _p(U_pred),
             U_pred.stride(0) if U_pred is not None else 0, _stream())
        return self.corr

    def backward(self, h, d_out, on_layer_grads=None):
        """dW / db of every layer into the flat gradient buffer; on_layer_grads(l) is called once dW / db of layer l are
        enqueued on the current stream (hook for the sharded engine's per-layer gradient all-reduce).  For each layer the dW kernel (side stream) and
        the dX kernel (main stream) run concurrently on half of the SMs each, walking the tiles in the same order:
        the dZ tile that one of them pulls from HBM is an L2 hit for the other, so dZ is read from DRAM once."""
        L = self.L
        main = torch.cuda.current_stream()
        side = self.side_stream
        pack_rows(d_out, self.pd[-1], out=self.dz_out)
        dz, dz_w = self.dz_out, self.pd[-1]
        # SMs for the dX kernel / for the dW kernel of a concurrent pair (dX moves slightly more bytes and has the
        # heavier epilogue: an even split lets dW finish early and leaves dX alone on half of the machine)
        n_dx = min(self.sm_count - 1, max(1, int(round(self.sm_count * self.dx_share))))
        n_dw = self.sm_count - n_dx
        for l in range(L - 1, -1, -1):
            act = self.acts[l - 1] if l > 0 else self.x0
            if l > 0:
                side.wait_stream(main)
                with torch.cuda.stream(side):
                    call("ep_tc_linear_dw_bf16", self.n, self.dims[l + 1], self.dims[l], dz_w, self.pd[l], _p(dz), _p(act),
                         _p(self.p.dW[l]), _p(self.p.db[l]), _p(self.ws), self.ws_bytes, n_dw, _stream())
                nxt = self.dz[l & 1]
                call("ep_tc_linear_dx_bf16", self.n, dz_w, self.pd[l], _p(dz), _p(self.WTp[l]), _p(self.masks[l - 1]),
                     _p(nxt), n_dx, _stream())
                main.wait_stream(side)
                dz, dz_w = nxt, self.pd[l]
            else:
                call("ep_tc_linear_dw_bf16", self.n, self.dims[l + 1], self.dims[l], dz_w, self.pd[l], _p(dz), _p(act),
                     _p(self.p.dW[l]), _p(self.p.db[l]), _p(self.ws), self.ws_bytes, 0, _stream())
            if on_layer_grads is not None:
                on_layer_grads(l)
