"""Weights of the SA path: initialisation in the reference's variable layout and inference-time folding.

Variable names follow the reference's TF scopes (SURVEY.md section 5; lib/utils/layers_util.py:175,185 and
lib/utils/tf_util.py:96,111,119):
  <scope>/conv{i}_{j}/weights [cin,cout]   (TF kernel [1,1,cin,cout] squeezed)
  <scope>/conv{i}_{j}/biases  [cout]
  <scope>/conv{i}_{j}/bn/{gamma,beta,moving_mean,moving_variance} [cout]
  <scope>/ensemble/...                      aggregation conv1d
  <scope>/vote_layer_{i}/..., <scope>/vote_offsets/...  (vote layer, layers_util.py:18-19)
"""
import numpy as np
import torch

from . import config as _cfg

FUSED_SMEM_LIMIT = 226 * 1024
BN_EPS = 1e-3  # tf.contrib.layers.batch_norm default epsilon (tf_util.py:439-444 does not override it)


def _conv_init(rng, params, scope, cin, cout, bn):
    limit = np.sqrt(6.0 / (cin + cout))  # tf.contrib.layers.xavier_initializer, uniform (tf_util.py:41)
    params[scope + "/weights"] = rng.uniform(-limit, limit, size=(cin, cout)).astype(np.float32)
    params[scope + "/biases"] = np.zeros((cout,), np.float32)  # tf_util.py:110
    if bn:  # randomised statistics so that the folding is actually exercised (SURVEY.md section 8d)
        params[scope + "/bn/gamma"] = rng.uniform(0.5, 1.5, size=(cout,)).astype(np.float32)
        params[scope + "/bn/beta"] = (0.1 * rng.standard_normal(cout)).astype(np.float32)
        params[scope + "/bn/moving_mean"] = (0.1 * rng.standard_normal(cout)).astype(np.float32)
        params[scope + "/bn/moving_variance"] = rng.uniform(0.5, 1.5, size=(cout,)).astype(np.float32)


def init_params(arch, in_channels, seed=0, random_bias=False):
    """Random weights for every conv of `arch` (numpy dict keyed by TF variable name)."""
    rng = np.random.default_rng(seed)
    params = {}
    ch = _cfg.layer_channels(arch, in_channels)
    for li, spec in enumerate(arch):
        (_, feat_i, radius, _, mlps, bn, _, _, _, _, _, ltype, scope, _, _, agg) = spec
        cin = ch[feat_i[0]]
        if ltype == "SA_Layer":
            if len(radius) == 0:
                continue
            for i, mlp in enumerate(mlps):
                c = cin + 3
                for j, cout in enumerate(mlp):
                    _conv_init(rng, params, "%s/conv%d_%d" % (scope, i, j), c, cout, bn)
                    c = cout
            if agg is not None and agg != -1 and _cfg.AGGREGATION_SA_FEATURE:
                _conv_init(rng, params, scope + "/ensemble", sum(m[-1] for m in mlps), agg, bn)
        elif ltype == "Vote_Layer":
            c = cin
            for i, cout in enumerate(mlps):
                _conv_init(rng, params, "%s/vote_layer_%d" % (scope, i), c, cout, bn)
                c = cout
            _conv_init(rng, params, scope + "/vote_offsets", c, 3, False)
        elif ltype == "SA_Layer_SSG_Last":
            c = cin + 3
            for j, cout in enumerate(mlps):
                _conv_init(rng, params, "%s/conv%d" % (scope, j), c, cout, bn)
                c = cout
        elif ltype == "FP_Layer":
            c = cin + ch[feat_i[1]] if len(feat_i) > 1 else cin
            for j, cout in enumerate(mlps):
                _conv_init(rng, params, "%s/conv_%d" % (scope, j), c, cout, bn)
                c = cout
    if random_bias:
        for k in list(params):
            if k.endswith("/biases"):
                params[k] = (0.1 * rng.standard_normal(params[k].shape)).astype(np.float32)
    return params


def round16(x):
    return (int(x) + 15) // 16 * 16


def init_head_params(cin, mlp=(128,), cls_channels=1, reg_channels=6 + 2 * 12, seed=1, scope=''):
    """Random weights of the detection head (head_builder.py:93-95, head_util.py:26-41) keyed by the reference's
    variable names: conv1d_{i}, pred_cls_base, pred_cls, pred_reg_base, pred_reg (scope '' in 3dssd.yaml:68)."""
    rng = np.random.default_rng(seed)
    pre = "" if scope == "" else scope + "/"
    params = {}
    c = cin
    for i, ch in enumerate(mlp):
        _conv_init(rng, params, "%sconv1d_%d" % (pre, i), c, ch, True)
        c = ch
    _conv_init(rng, params, pre + "pred_cls_base", c, 128, True)
    _conv_init(rng, params, pre + "pred_cls", 128, cls_channels, False)
    _conv_init(rng, params, pre + "pred_reg_base", c, 128, True)
    _conv_init(rng, params, pre + "pred_reg", 128, reg_channels, False)
    for k in list(params):
        if k.endswith("/biases"):
            params[k] = (0.1 * rng.standard_normal(params[k].shape)).astype(np.float32)
    return params


class FoldedConv:
    """One conv+BN layer folded for inference: y = act((x @ w) * scale + shift).
    For the tensor-core path the weight also exists split in two bf16 terms, transposed to K-major:
    b_hi + b_lo ~= w^T, shape [cout, kp] with kp = round16(cin) (zero padded)."""
    __slots__ = ("w", "scale", "shift", "cin", "cout", "kp", "b_hi", "b_lo")

    def __init__(self, w, scale, shift):
        self.w, self.scale, self.shift = w, scale, shift
        self.cin, self.cout = w.shape
        self.kp = round16(self.cin)
        wt = torch.zeros((self.cout, self.kp), dtype=torch.float32, device=w.device)
        wt[:, : self.cin] = w.t()
        self.b_hi = wt.to(torch.bfloat16)                       # round-to-nearest-even, like the device split
        self.b_lo = (wt - self.b_hi.to(torch.float32)).to(torch.bfloat16)

    def __repr__(self):
        return "FoldedConv(%d -> %d)" % (self.cin, self.cout)


def fold(params, scope, bn, device):
    """inv = gamma * rsqrt(var + eps);  y = (xW + b) * inv + (beta - mean * inv)   (tf_util.py:439-444)."""
    w = np.asarray(params[scope + "/weights"], np.float64)
    b = np.asarray(params.get(scope + "/biases", np.zeros(w.shape[1])), np.float64)
    if bn:
        g = np.asarray(params[scope + "/bn/gamma"], np.float64)
        be = np.asarray(params[scope + "/bn/beta"], np.float64)
        mu = np.asarray(params[scope + "/bn/moving_mean"], np.float64)
        var = np.asarray(params[scope + "/bn/moving_variance"], np.float64)
        inv = g / np.sqrt(var + BN_EPS)
        scale, shift = inv, (b - mu) * inv + be
    else:
        scale, shift = np.ones_like(b), b
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(device)
    return FoldedConv(t(w), t(scale), t(shift))


def _k_blocks(kp):
    """Operand layout of the fused kernel for a padded K: (nfull, rbt) = number of 64-wide k-blocks (128-byte rows) and
    the row bytes of the tail block -- 0 / 32 / 64 / 128 for a remainder of 0 / 16 / 32 / 48 columns (must match
    sf_rbt_of in csrc/sa_fused.cu)."""
    rem = kp % 64
    return kp // 64, 0 if rem == 0 else (32 if rem <= 16 else (64 if rem <= 32 else 128))


def _swizzle_block(blk, rb):
    """[npad, rb/2] bf16 -> canonical UMMA K-major image with swizzle span rb: 16-byte chunk j of row r is stored at
    chunk j ^ ((r >> log2(128/rb)) & (rb/16 - 1)), i.e. SWIZZLE_128B / _64B / _32B for rb = 128 / 64 / 32."""
    npad = blk.shape[0]
    nc = rb // 16
    sh = {128: 0, 64: 1, 32: 2}[rb]
    t = blk.reshape(npad, nc, 8)
    r = torch.arange(npad, device=blk.device).view(npad, 1, 1)
    j = torch.arange(nc, device=blk.device).view(1, nc, 1)
    src = (j ^ ((r >> sh) & (nc - 1))).expand(npad, nc, 8)
    return torch.gather(t, 1, src).contiguous().view(-1)


def _swizzled_image(wt_bf16):
    """[npad, kp] bf16 (W^T, K-major) -> the fused kernel's operand image: nfull blocks of [npad x 128 bytes] followed
    by the tail block of [npad x rbt bytes] (zero padded), each block swizzled over its own row span."""
    npad, kp = wt_bf16.shape
    nfull, rbt = _k_blocks(kp)
    parts = [_swizzle_block(wt_bf16[:, 64 * i: 64 * (i + 1)].contiguous(), 128) for i in range(nfull)]
    if rbt:
        tail = torch.zeros((npad, rbt // 2), dtype=torch.bfloat16, device=wt_bf16.device)
        tail[:, : kp - 64 * nfull] = wt_bf16[:, 64 * nfull:]
        parts.append(_swizzle_block(tail, rbt))
    return torch.cat(parts)


class FusedStack:
    """Operands of ssd3d_sa_mlp_fused for one SA scale: the split, pre-swizzled weight images of its conv layers
    packed as { hi | lo } per layer, and the folded { scale | shift } per layer (zero beyond the true width)."""

    def __init__(self, convs, cin):
        dev = convs[0].w.device
        self.nout = [f.cout for f in convs]
        self.cin = cin
        self.convs = list(convs)            # the folded layers the blobs were built from (introspection / CPU dry runs)
        # The LAST layer is stored with non-negative scales: (x.w) * s + t == (x.(w * sgn s)) * |s| + t, exactly (a sign
        # flip is exact in bf16).  fma(acc, |s|, t) is then monotone in acc, so the kernel may max-pool the raw
        # accumulators and apply scale / shift / ReLU to the pooled values only (ssd3d.h: last_scale_nonneg).
        self.last_scale_nonneg = True
        wparts, sparts = [], []
        kp = round16(cin)
        for li, f in enumerate(convs):
            npad = round16(f.cout)
            assert f.kp == kp, (f.kp, kp)
            b_hi, b_lo, scale = f.b_hi, f.b_lo, f.scale
            if li == len(convs) - 1:
                sgn = torch.where(scale < 0, -torch.ones_like(scale), torch.ones_like(scale))
                b_hi = (b_hi.float() * sgn.unsqueeze(1)).to(torch.bfloat16)
                b_lo = (b_lo.float() * sgn.unsqueeze(1)).to(torch.bfloat16)
                scale = scale.abs()
            hi = torch.zeros((npad, kp), dtype=torch.bfloat16, device=dev)
            lo = torch.zeros_like(hi)
            hi[: f.cout] = b_hi
            lo[: f.cout] = b_lo
            wparts += [_swizzled_image(hi), _swizzled_image(lo)]
            sspad = (npad + 31) // 32 * 32                 # the kernel reads scale/shift in 32-column chunks
            sc = torch.zeros(sspad, dtype=torch.float32, device=dev)
            sh = torch.zeros(sspad, dtype=torch.float32, device=dev)
            sc[: f.cout] = scale
            sh[: f.cout] = f.shift
            sparts += [sc, sh]
            kp = npad
        self.w_blob = torch.cat(wparts).contiguous()
        self.ss_blob = torch.cat(sparts).contiguous()

    def __repr__(self):
        return "FusedStack(%d -> %s)" % (self.cin, self.nout)


class PreparedParams:
    """Device-resident folded weights, looked up by TF scope name (lazy, cached)."""

    def __init__(self, params, device):
        self.raw = params
        self.device = torch.device(device)
        self._cache = {}

    def conv(self, scope, bn=True):
        key = (scope, bool(bn))
        if key not in self._cache:
            self._cache[key] = fold(self.raw, scope, bn, self.device)
        return self._cache[key]

    def fused_stack(self, scopes, bn, cin, limit=None):
        """FusedStack for a list of conv scopes (one SA scale), or None when the stack does not fit the fused kernel
        (limit = shared-memory bytes the policy allows; default FUSED_SMEM_LIMIT, pass 0 for 'whatever fits')."""
        limit = FUSED_SMEM_LIMIT if limit is None else (limit or 1 << 30)
        key = ("fused",) + tuple(scopes) + (bool(bn), cin, limit)
        if key not in self._cache:
            import ctypes
            from ._lib import lib
            convs = [self.conv(sc, bn) for sc in scopes]
            nout = (ctypes.c_int * len(convs))(*[f.cout for f in convs])
            need = lib().ssd3d_sa_fused_smem(cin - 3, len(convs), ctypes.cast(nout, ctypes.c_void_p)) if len(convs) <= 3 else 0
            # the fused kernel keeps every layer's weights in shared memory; stacks that do not fit (layer3/4 sized)
            # return None and take the layer-by-layer tensor-core path
            fits = 0 < need <= limit
            self._cache[key] = FusedStack(convs, cin) if fits else None
        return self._cache[key]

    def hoisted(self, scopes, bn, c):
        """First convs of the scales of one SA layer (scopes), hoisted: returns (FoldedConv for the per-point table
        z = (f . [Wf_1 | Wf_2 | ...]) * s + t over all scales, [Wx_i * s_i as (3, n1_i) per scale], [n1_i]).
        c = feature channels (the convs take c + 3 inputs: features first, then xyz - centre)."""
        key = ("hoisted",) + tuple(scopes) + (bool(bn), c)
        if key not in self._cache:
            convs = [self.conv(sc, bn) for sc in scopes]
            for f in convs:
                if f.cin != c + 3:
                    raise ValueError("hoisted: conv expects %d inputs, got c + 3 = %d" % (f.cin, c + 3))
            wf = torch.cat([f.w[:c] for f in convs], dim=1).contiguous()
            zconv = FoldedConv(wf, torch.cat([f.scale for f in convs]).contiguous(), torch.cat([f.shift for f in convs]).contiguous())
            wxs = [(f.w[c:c + 3].double() * f.scale.double().unsqueeze(0)).float().contiguous() for f in convs]
            self._cache[key] = (zconv, wxs, [f.cout for f in convs])
        return self._cache[key]

    # ---- training mode: BatchNorm state lives on the device and is updated in place by the forward -----------------
    def bn_state(self, scope):
        """{gamma, beta, moving_mean, moving_variance} of `scope` as device tensors; training-mode forwards update the
        moving statistics in place.  commit_bn() writes them back to the parameter dict."""
        key = ("bn_state", scope)
        if key not in self._cache:
            self._cache[key] = {k: torch.from_numpy(np.ascontiguousarray(self.raw[scope + "/bn/" + k], dtype=np.float32)).to(self.device)
                                for k in ("gamma", "beta", "moving_mean", "moving_variance")}
        return self._cache[key]

    def commit_bn(self):
        """Copy the moving statistics updated by training-mode forwards back into the raw parameter dict and drop every
        folded form derived from the old ones (inference after training folds the new statistics)."""
        touched = False
        for key in [k for k in self._cache if isinstance(k, tuple) and k[0] == "bn_state"]:
            st = self._cache[key]
            for k in ("moving_mean", "moving_variance"):
                self.raw[key[1] + "/bn/" + k] = st[k].detach().cpu().numpy()
            touched = True
        if touched:
            for key in [k for k in self._cache if not (isinstance(k, tuple) and k[0] == "bn_state")]:
                del self._cache[key]
        return self

    def prepare_all(self):
        for k in self.raw:
            if k.endswith("/weights"):
                scope = k[: -len("/weights")]
                self.conv(scope, (scope + "/bn/gamma") in self.raw)
        return self


def prepare(params, device="cuda"):
    return params if isinstance(params, PreparedParams) else PreparedParams(params, device)
