"""DecoderPlan: flattens a DeepSDF ``Decoder`` into the device buffers libdist_b200.so consumes.

What is folded away here (once per weight version, not once per decoder call as in the reference):
  * weight normalisation  W = g * v / ||v||      (deep_sdf_decoder.py:59, recomputed by a forward pre-hook there)
  * the latent code: layer 0 becomes K=3 (xyz) and the ``latent_in`` layer K = h + 3, the latent contribution
    being a per-render bias  b' = b + W[:, latent cols] @ z  (dist_fold_latent)   -- SURVEY.md section 7 step 2.
Weights are read from the live module; the plan re-flattens itself when a parameter's version counter changes
(e.g. after an optimizer step on the decoder).
"""
import torch

from . import _abi


def _round_up(x, m):
    return (x + m - 1) // m * m


def effective_linear(lin):
    """(weight[out,in], bias[out]) of a (possibly weight-normalised) linear layer, fp32."""
    if hasattr(lin, "weight_g") and hasattr(lin, "weight_v"):
        w = torch._weight_norm(lin.weight_v, lin.weight_g, 0)
    elif hasattr(lin, "parametrizations") and hasattr(lin.parametrizations, "weight"):
        w = lin.weight
    else:
        w = lin.weight
    return w.detach().float(), lin.bias.detach().float()


class DecoderPlan(object):
    def __init__(self, decoder):
        self.decoder = decoder
        self._key = None
        self.refresh()

    # ---- validation of the network family the kernels cover
    def _validate(self):
        d = self.decoder
        n_lin = d.num_layers - 1
        if n_lin < 2 or n_lin > _abi.MAX_LAYERS:
            raise NotImplementedError("decoder with %d linear layers is outside the fused path [2,%d]"
                                      % (n_lin, _abi.MAX_LAYERS))
        if getattr(d, "xyz_in_all", None):
            raise NotImplementedError("xyz_in_all decoders are not supported by the fused path")
        if (not getattr(d, "weight_norm", False)) and d.norm_layers is not None and len(d.norm_layers) > 0:
            raise NotImplementedError("LayerNorm decoders (norm_layers without weight_norm) are not supported")
        if getattr(d, "latent_dropout", False) and d.training:
            raise NotImplementedError("latent dropout in training mode is not supported")
        if d.training and d.dropout is not None and len(d.dropout) > 0 and d.dropout_prob > 0:
            raise NotImplementedError("decoder must be in eval() mode (dropout is not implemented)")
        lat_in = list(d.latent_in) if d.latent_in is not None else []
        if len(lat_in) > 1:
            raise NotImplementedError("more than one latent_in layer is not supported")
        if lat_in and not (1 <= lat_in[0] < n_lin - 1):
            raise NotImplementedError("latent_in must name a hidden layer >= 1")

    def _version_key(self):
        return tuple((p.data_ptr(), p._version) for p in self.decoder.parameters())

    def refresh(self, force=False):
        key = self._version_key()
        if not force and key == self._key:
            return False
        self._validate()
        d = self.decoder
        dev = next(d.parameters()).device
        if dev.type != "cuda":
            raise ValueError("the decoder must live on a CUDA device (no CPU path)")
        self.device = dev
        n_lin = d.num_layers - 1
        self.n_layers = n_lin
        lat_in = list(d.latent_in) if d.latent_in is not None else []
        self.latent_in = lat_in[0] if lat_in else -1
        first_w, _ = effective_linear(getattr(d, "lin0"))
        self.latent_size = first_w.shape[1] - 3
        Lz = self.latent_size
        self.K, self.N, self.Wt, self.W, self.bias = [], [], [], [], []
        self.Wz0 = self.b0 = self.Wzl = self.bl = None
        prev = None
        for l in range(n_lin):
            w, b = effective_linear(getattr(d, "lin%d" % l))
            n_out, n_in = w.shape
            if l == 0:
                self.Wz0, self.b0 = w[:, :Lz].contiguous(), b.contiguous()
                wf = w[:, Lz:Lz + 3]
            elif l == self.latent_in:
                h = n_in - (Lz + 3)
                if h != prev:
                    raise NotImplementedError("latent_in layer input width mismatch")
                self.Wzl, self.bl = w[:, h:h + Lz].contiguous(), b.contiguous()
                wf = torch.cat([w[:, :h], w[:, h + Lz:h + Lz + 3]], 1)
            else:
                wf = w
                if n_in != prev:
                    raise NotImplementedError("layer %d input width %d != previous output %d" % (l, n_in, prev))
            k = wf.shape[1]
            if max(k, n_out) > _abi.MAX_WIDTH:
                raise NotImplementedError("layer width > %d is not supported" % _abi.MAX_WIDTH)
            wt = torch.zeros(_round_up(k, 8), _round_up(n_out, 4), device=dev)
            wt[:k, :n_out] = wf.t()
            wn = torch.zeros(_round_up(n_out, 8), _round_up(k, 4), device=dev)
            wn[:n_out, :k] = wf
            bp = torch.zeros(_round_up(n_out, 4), device=dev)
            bp[:n_out] = b
            self.K.append(k); self.N.append(n_out)
            self.Wt.append(wt); self.W.append(wn); self.bias.append(bp)
            prev = n_out
        # The kernels evaluate ONE output per launch (dot product + tanh in the epilogue).  A decoder with several outputs
        # (the colour network of renderer_rgb.py:20-38, last_dim = 3) is evaluated as n_out single-output networks that
        # share every hidden layer: c_net(out_index=c) points the last layer at row c of its weights.
        self.n_out = self.N[-1]
        if self.n_out > 4:
            raise NotImplementedError("decoders with more than 4 outputs are not supported by the fused path")
        self.use_tanh = 1 if getattr(d, "use_tanh", False) else 0
        self.tc = None      # tensor-core operand blobs, built lazily by tc.prepare()
        self.tc_unsafe = False
        self._key = key
        return True

    def fold(self, latent, stream, n_codes=1):
        """Per-render folded biases (device tensors) for layer 0 and the latent_in layer.  With n_codes = C > 1, `latent`
        holds C codes (C, L) and the biases are per-code tables, flat [C][Np4]: row c is byte for byte what folding code c
        alone gives (one launch, the codes on the grid's second dimension)."""
        lib = _abi.lib()
        C = max(1, int(n_codes))
        f32 = dict(device=self.device, dtype=torch.float32)
        out0 = torch.empty(C * self.bias[0].numel(), **f32)
        outl = torch.empty(C * self.bias[self.latent_in].numel(), **f32) if self.latent_in >= 0 else None
        net = self.c_net(None, None, n_codes=C)
        lat = None
        if self.latent_size > 0:
            if latent is None:
                raise ValueError("this decoder expects a latent code")
            lat = latent.detach().reshape(-1).float().contiguous()
            if lat.numel() != C * self.latent_size:
                raise ValueError("latent has %d elements, decoder expects %d" % (lat.numel(), C * self.latent_size))
        _abi.check(lib.dist_fold_latent(net, _abi.ptr(lat), _abi.ptr(out0), _abi.ptr(outl), stream))
        return out0, outl, lat

    def net_for(self, latent, engine, stream, out_index=0, n_codes=1):
        """(dist_net_t, effective engine, keepalive) for one call: prepares the tensor-core operands when that engine is selected,
        folds the latent into the per-render biases and fills the descriptor (for output `out_index` of the network).
        n_codes > 1: `latent` is (n_codes, L) and the descriptor carries per-code bias tables (dist_net_t.n_codes); the caller
        says which code each row uses (dist_net_t.row_code, or the view of the pixel in a render)."""
        if engine == _abi.ENGINE_TC:
            from . import tc
            try:
                tc.prepare(self)
            except NotImplementedError:
                if not getattr(self, "tc_unsafe", False):
                    raise
                engine = _abi.ENGINE_SIMT       # self-check failed (warned once): this call runs on the fp32 engine
        b0, bl, lat = self.fold(latent, stream, n_codes)
        bl_tc = None
        if engine == _abi.ENGINE_TC and bl is not None:
            from . import tc
            bl_tc = bl * tc.S_ACT
        net = self.c_net(b0, bl, bl_tc, out_index=out_index, n_codes=n_codes)
        return net, engine, (b0, bl, bl_tc, lat)

    def c_net(self, bias0, biasl, biasl_tc=None, out_index=0, n_codes=1):
        """ctypes dist_net_t for one call; bias0/biasl are the folded biases (or None before folding); `out_index` selects
        which output of a multi-output network the (single-output) kernels compute; n_codes > 1: bias0/biasl are per-code
        tables (dist_net_t.n_codes)."""
        if not (0 <= out_index < self.n_out):
            raise ValueError("out_index %d outside the decoder's %d outputs" % (out_index, self.n_out))
        net = _abi.Net()
        net.n_layers, net.latent_size, net.latent_in, net.use_tanh = self.n_layers, self.latent_size, \
            self.latent_in, self.use_tanh
        net.n_codes = int(n_codes) if n_codes > 1 else 0
        for l in range(self.n_layers):
            net.K[l], net.N[l] = self.K[l], self.N[l]
            net.Wt[l], net.W[l] = self.Wt[l].data_ptr(), self.W[l].data_ptr()
            b = self.bias[l]
            if l == 0 and bias0 is not None:
                b = bias0
            if l == self.latent_in and biasl is not None:
                b = biasl
            net.bias[l] = b.data_ptr()
        last = self.n_layers - 1
        net.N[last] = 1
        net.W[last] = self.W[last].data_ptr() + 4 * out_index * self.W[last].shape[1]      # row out_index of [Np8][Kp4]
        net.bias[last] = self.bias[last].data_ptr() + 4 * out_index
        net.Wz0 = self.Wz0.data_ptr() if self.Wz0 is not None and self.Wz0.numel() else None
        net.b0 = self.b0.data_ptr()
        if self.latent_in >= 0:
            net.Wzl, net.bl = self.Wzl.data_ptr(), self.bl.data_ptr()
        if self.tc is not None:
            import ctypes
            net.tc_blob = self.tc["blob"].data_ptr()
            net.tc_scale = ctypes.addressof(self.tc["inv_scale"])
            net.tc_blob_bytes = self.tc["blob"].numel() * self.tc["blob"].element_size()
            for l in range(self.n_layers):
                b = self.tc["bias_s"][l]
                if l == self.latent_in and biasl_tc is not None:
                    b = biasl_tc
                net.tc_bias[l] = b.data_ptr()
        return net

    def latent_grad(self, acc0, accl, n_codes=1):
        """dL/dlatent from the accumulated pre-activation gradients of layer 0 and the latent_in layer: (1, L), or (C, L)
        from the per-code accumulators [C][N] of a call with n_codes = C > 1."""
        if n_codes > 1:
            C = int(n_codes)
            g = acc0[: C * self.N[0]].reshape(C, self.N[0]) @ self.Wz0
            if self.latent_in >= 0:
                g = g + accl[: C * self.N[self.latent_in]].reshape(C, self.N[self.latent_in]) @ self.Wzl
            return g
        g = acc0[: self.N[0]] @ self.Wz0
        if self.latent_in >= 0:
            g = g + accl[: self.N[self.latent_in]] @ self.Wzl
        return g.reshape(1, -1)

    def acc_buffers(self, n_codes=1):
        """Zeroed accumulators acc0 / accl of a backward call: [Np4] (one code, as always) or [n_codes][N]."""
        if n_codes > 1:
            n0, nl = n_codes * self.N[0], (n_codes * self.N[self.latent_in] if self.latent_in >= 0 else 0)
        else:
            n0, nl = self.bias[0].numel(), (self.bias[self.latent_in].numel() if self.latent_in >= 0 else 0)
        acc0 = torch.zeros(n0, device=self.device, dtype=torch.float32)
        accl = torch.zeros(nl, device=self.device, dtype=torch.float32) if self.latent_in >= 0 else None
        return acc0, accl


_PLANS = {}


def plan_for(decoder):
    """One cached plan per decoder object, refreshed when its weights change."""
    p = _PLANS.get(id(decoder))
    if p is None or p.decoder is not decoder:
        p = DecoderPlan(decoder)
        _PLANS[id(decoder)] = p
    else:
        p.refresh()
    return p
