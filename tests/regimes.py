"""Value regimes for the gradient tests: where the GRU gates saturate and the logits are peaked.

At the reference's default init (oracle.init_params) and the synthetic features of make_batch, the GRU pre-activations
are small: z and r stay near 0.5, |h_hat| stays far below 1 and the logits span about +-1.  The backward rebuilds
z (1 - z), 1 - z and 1 - h_hat^2 from bf16-stashed gates and the loss kernels rescale per-tile softmax statistics; at
that point neither has any effect a test could see.  Each constructor below takes init_params output plus a batch
(feat_v, feat_n, gt_verb, gt_nouns) and returns modified parameters and inputs that move the model to one of the
value regimes a trained model reaches.  tests/test_saturation.py checks on the fp64 oracle that every regime is what
it claims to be and that a saturation-only bug is visible in it; tests/test_saturation_gpu.py runs the CUDA paths there.

Plain helper module (no tests); everything runs on the device and in the dtype of the tensors passed in.
"""
import contextlib

import torch
import torch.nn.functional as F

from oracle import ggnn_oracle as O

GATES = ("W_z", "U_z", "W_r", "U_r", "W_h", "U_h")
GGSNN_KEYS = tuple("ggsnn.%s.%s" % (k, w) for k in O.GGNN_KEYS for w in ("weight", "bias"))
NUM_LABELS = 2001


def tables(enc):
    return O.build_tables(enc.roles_per_verb, enc.verb_list, enc.role_list)


def random_mask(B, R, seed):
    """Asymmetric, real-valued, with self-loops, exact zeros and an all-zero row in every third image."""
    g = torch.Generator().manual_seed(seed)
    mk = torch.rand(B, R, R, generator=g) * 2 - 1
    mk[torch.rand(B, R, R, generator=g) < 0.25] = 0.0
    mk[::3, R // 2, :] = 0.0
    return mk


# ---------------------------------------------------------------------------------------------- regimes
def init(params, batch, tabs):
    """The control: the suite's usual point, unchanged."""
    return dict(params), batch


def gates_x8(params, batch, tabs):
    """The six gate matrices (W / U of z, r, h) x 8: both tails of z and r, and saturated h_hat."""
    p = dict(params)
    for k in GATES:
        p["ggsnn.%s.weight" % k] = params["ggsnn.%s.weight" % k] * 8
    return p, batch


def gate_bias(params, batch, tabs):
    """U_z and U_r biases = +4 on the first half of the columns and -4 on the second: z ~ 1 (overwrite) columns next
    to z ~ 0 (carry) columns."""
    p = dict(params)
    for k in ("U_z", "U_r"):
        b = torch.full_like(params["ggsnn.%s.bias" % k], 4.0)
        b[b.shape[0] // 2:] = -4.0
        p["ggsnn.%s.bias" % k] = b
    return p, batch


PEAK_SCALE = 512.0


def peaked(params, batch, tabs):
    """Both classifiers (weights and biases) x PEAK_SCALE: softmaxes close to one-hot.  The targets of every other
    image are set to the oracle's own argmax (verb, and every scored role of the predicted-verb noun path), so the
    losses see rows whose target is the top-1 next to rows whose target is far down the ranking."""
    p = dict(params)
    for k in ("verb_classifier.1", "nouns_classifier.1"):
        for w in ("weight", "bias"):
            p["%s.%s" % (k, w)] = params["%s.%s" % (k, w)] * PEAK_SCALE
    fv, fn, gt_verb, gt_nouns = batch
    t, c = tabs
    with torch.no_grad():
        pv = O.predict_verb(p, fv)
        gt_verb = gt_verb.clone()
        gt_verb[::2] = pv.argmax(-1)[::2].to(gt_verb.device)
        pn = O.predict_nouns(p, fn, pv.argmax(-1), t, c)
    # the even images' verbs changed: their role slots are re-derived (pad slots get the ignore label)
    top = pn.argmax(-1)[::2].to(gt_nouns.device)
    scored = torch.arange(t.shape[1])[None, :] < torch.from_numpy(c[gt_verb[::2].cpu().numpy()])[:, None]
    gt_nouns = gt_nouns.clone()
    gt_nouns[::2] = torch.where(scored.to(gt_nouns.device), top, NUM_LABELS)[:, None, :]
    return p, (fv, fn, gt_verb, gt_nouns)


def fitted(params, batch, tabs, lr=0.01, max_steps=300, target=1.0):
    """A real trained point: Adamax (gradient norm clipped to 1, as the launcher) on one batch whose three noun
    annotations agree, with the oracle's fp32 step, until verb_loss + nouns_loss < target."""
    fv, fn, gt_verb, gt_nouns = batch
    gt_nouns = gt_nouns[:, :1].expand(-1, 3, -1).contiguous()
    t, c = tabs
    ps = {k: v.detach().clone().float().requires_grad_(True) for k, v in params.items()}
    opt = torch.optim.Adamax(list(ps.values()), lr=lr)
    dv, dn = gt_verb.to(fv.device), gt_nouns.to(fv.device)
    for _ in range(max_steps):
        opt.zero_grad()
        pv = O.predict_verb(ps, fv.float())
        pn = O.predict_nouns(ps, fn.float(), pv.argmax(-1), t, c)
        loss = O.verb_loss(pv, dv) + O.nouns_loss(pn, dn, NUM_LABELS)
        if loss.item() < target:
            break
        loss.backward()
        torch.nn.utils.clip_grad_norm_(list(ps.values()), 1.0)
        opt.step()
    else:
        raise RuntimeError("fitted: the loss is still %.3f after %d steps" % (loss.item(), max_steps))
    p = {k: v.detach().to(params[k].dtype) for k, v in ps.items()}
    return p, (fv, fn, gt_verb, gt_nouns)


def big_states(params, hidden, mask):
    """model.ggsnn only: node states x 10 and the (random, real-valued) adjacency mask x 3."""
    return dict(params), hidden * 10, (None if mask is None else mask * 3)


REGIMES = {"init": init, "gates_x8": gates_x8, "gate_bias": gate_bias, "peaked": peaked, "fitted": fitted}


# ---------------------------------------------------------------------------------------------- oracle helpers
def gate_trace(params, batch, tabs, verbs=None):
    """z, r and h_hat of every GRU step of the verb path and of the noun path (conditioned on `verbs`, default the gt
    verbs), flattened: {"verb": {...}, "nouns": {...}}."""
    fv, fn, gt_verb, _ = batch
    t, c = tabs
    p = O._sub(params, "ggsnn.")
    verbs = gt_verb if verbs is None else verbs
    out = {}
    with torch.no_grad():
        tr = []
        O.ggsnn_forward(p, F.relu(fv), verb=True, trace=tr)
        out["verb"] = _flat(tr)
        B, R = fn.shape[0], t.shape[1]
        role_idx = torch.from_numpy(O.get_role_ids_batch(t, verbs.cpu().numpy())).to(fn.device)
        node = F.relu(fn[:, None] * params["role_emb.weight"][role_idx] *
                      params["verb_emb.weight"][verbs.to(fn.device)][:, None]).reshape(B * R, -1)
        mask = torch.from_numpy(O.get_adj_matrix_noself(c, verbs.cpu().numpy(), R)).to(fn.device, fn.dtype)
        tr = []
        O.ggsnn_forward(p, node, mask=mask, trace=tr)
        out["nouns"] = _flat(tr)
    return out


def _flat(tr):
    return {k: torch.cat([s[k].flatten() for s in tr]) for k in ("z", "r", "h_hat")}


def gate_stats(g):
    """Fractions of the gate values in the saturated tails (inputs of the coverage assertions)."""
    return {"z_low": float((g["z"] < 0.1).double().mean()), "z_high": float((g["z"] > 0.9).double().mean()),
            "r_low": float((g["r"] < 0.1).double().mean()), "r_high": float((g["r"] > 0.9).double().mean()),
            "h_hat_sat": float((g["h_hat"].abs() > 0.9).double().mean())}


def oracle_step(params, batch, tabs, pred_verbs=None, keeps=(None, None, None), feat_grad=False,
                dtype=torch.float64, device="cpu", num_labels=NUM_LABELS):
    """sr.py's training step (verb_loss + nouns_loss of the predicted-verb path) under fp64 autograd of the oracle;
    num_labels is the vocabulary size, the noun targets' ignore label.
    Returns (losses (verb, nouns, gt nouns), {param: grad}, logits (verb, pred nouns, gt nouns), (dfeat_v, dfeat_n))."""
    fv, fn, gt_verb, gt_nouns = batch
    t, c = tabs
    ps = {k: v.detach().to(device, dtype).clone().requires_grad_(True) for k, v in params.items()}
    xv = fv.detach().to(device, dtype).clone().requires_grad_(feat_grad)
    xn = fn.detach().to(device, dtype).clone().requires_grad_(feat_grad)
    kp = tuple(None if k is None else k.to(device) for k in keeps)
    gv, gn = gt_verb.to(device), gt_nouns.to(device)
    pv, pn, gpn = O.forward(ps, xv, xn, gv, t, c, kp, 0.5, None if pred_verbs is None else pred_verbs.to(device))
    vl, nl, gl = O.verb_loss(pv, gv), O.nouns_loss(pn, gn, num_labels), O.nouns_loss(gpn, gn, num_labels)
    (vl + nl).backward()
    grads = {k: (v.grad if v.grad is not None else torch.zeros_like(v)) for k, v in ps.items()}
    return ((vl.detach(), nl.detach(), gl.detach()), grads, (pv.detach(), pn.detach(), gpn.detach()),
            (xv.grad, xn.grad))


def oracle_ggsnn(params, hidden, mask, G, dtype=torch.float64, device="cpu"):
    """fp64 autograd of the oracle's GGSNN for loss = (out * G).sum(): (out, d hidden, d mask or None, {name: grad})
    with the names of model.ggsnn's parameters."""
    ps = {k: v.detach().to(device, dtype).clone().requires_grad_(True) for k, v in O._sub(params, "ggsnn.").items()}
    h = hidden.detach().to(device, dtype).clone().requires_grad_(True)
    mk = None if mask is None else mask.detach().to(device, dtype).clone().requires_grad_(True)
    out = O.ggsnn_forward(ps, h, mask=mk, verb=mask is None)
    (out * G.to(device, dtype)).sum().backward()
    return out.detach(), h.grad, (None if mk is None else mk.grad), {k: v.grad for k, v in ps.items()}


# ---------------------------------------------------------------------------------------------- derivative variants
def _derivative_function(grad_of_output, fn):
    class Act(torch.autograd.Function):
        @staticmethod
        def forward(ctx, x):
            y = fn(x)
            ctx.save_for_backward(y)
            return y

        @staticmethod
        def backward(ctx, g):
            (y,) = ctx.saved_tensors
            return g * grad_of_output(y)

    return Act.apply


def _bf16(x):
    return x.to(torch.bfloat16).to(x.dtype)


def _bf16_folded(y):
    m = _bf16(torch.minimum(y, 1 - y))      # r folded to min(r, 1 - r), stashed in bf16 (gate_fold in gemm.cuh)
    return m * (1 - m)


# (derivative of z = sigmoid, of r = sigmoid, of h_hat = tanh), each as a function of the output
DERIVATIVES = {
    # a backward-only bug: the derivative factors are taken of z, r clamped to [0.05, 0.95] and of h_hat clamped to
    # [-0.95, 0.95]; the forward is unchanged
    "clamped": (lambda y: y.clamp(0.05, 0.95) * (1 - y.clamp(0.05, 0.95)),) * 2 +
               (lambda y: 1 - y.clamp(-0.95, 0.95) ** 2,),
    # the designed rounding of the per-step stash (DESIGN.md section 3): z (1 - z) and 1 - h_hat^2 rebuilt from bf16 z
    # and h_hat, r (1 - r) from the folded bf16 r
    "bf16_stash": (lambda y: _bf16(y) * (1 - _bf16(y)), _bf16_folded, lambda y: 1 - _bf16(y) ** 2),
}


@contextlib.contextmanager
def derivative(kind):
    """Within the block the oracle's GRU activations (oracle.gate_z, gate_r, candidate: names in the oracle's own
    module) keep their forward but back-propagate DERIVATIVES[kind] of their output."""
    saved = O.gate_z, O.gate_r, O.candidate
    dz, dr, dh = DERIVATIVES[kind]
    O.gate_z = _derivative_function(dz, torch.sigmoid)
    O.gate_r = _derivative_function(dr, torch.sigmoid)
    O.candidate = _derivative_function(dh, torch.tanh)
    try:
        yield
    finally:
        O.gate_z, O.gate_r, O.candidate = saved


class _Bf16Linear(torch.autograd.Function):
    """x @ w^T + b with both GEMM operands rounded to bf16, in the forward and in both backward GEMMs (the incoming
    gradient is a bf16 operand too), accumulated in the tensors' own dtype: the operand rounding of the CUDA path."""

    @staticmethod
    def forward(ctx, x, w, b):
        xb, wb = _bf16(x), _bf16(w)
        ctx.save_for_backward(xb, wb)
        return xb @ wb.t() + b

    @staticmethod
    def backward(ctx, g):
        xb, wb = ctx.saved_tensors
        gb = _bf16(g)
        g2, x2 = gb.reshape(-1, gb.shape[-1]), xb.reshape(-1, xb.shape[-1])
        return gb @ wb, g2.t() @ x2, g.reshape(-1, g.shape[-1]).sum(0)


@contextlib.contextmanager
def bf16_emulation():
    """The oracle with the designed rounding of the CUDA bf16 path: bf16 GEMM operands everywhere (oracle.linear) and
    the derivative factors rebuilt from the bf16 stash (DERIVATIVES["bf16_stash"]).  It does not reproduce the CUDA
    path's exact roundings (folded weights, summation order, tanh.approx), only their size."""
    saved = O.linear
    O.linear = _Bf16Linear.apply
    try:
        with derivative("bf16_stash"):
            yield
    finally:
        O.linear = saved


def relmax(a, b):
    """max |a - b| / max |b|: the suite's error metric (element-wise relative error is meaningless near zero)."""
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-300)).item()


def relfro(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return ((a - b).norm() / b.norm().clamp_min(1e-300)).item()
