"""CPU oracle for the GGNN role-graph stage of vFones/situation-recognition.

TEST INFRASTRUCTURE ONLY.  This is a from-scratch restatement (torch CPU / numpy, fp32 or fp64) of the
reference algorithm, function by function, each citing the reference file:line it follows.  Only `tests/`,
`__graft_entry__.smoke()` and the `cpu_baseline` / `--impl reference` legs of `bench.py` may import it; the
product path (situation_recognition_b200/) never does and fails loudly without its CUDA library.

Parity pinning: the reference ships no tests or golden vectors (SURVEY.md section 4), so this oracle is pinned
against the reference ITSELF, executed in the build container: `oracle/make_golden.py` imports the unmodified
`/root/reference/model.py` + `utils/imsitu_encoder.py`, runs them on seeded inputs and writes
`tests/golden/*.npz`; `tests/test_oracle_golden.py` checks every function below against those files.

The arithmetic is written AS THE REFERENCE WRITES IT (e.g. the [B,6,6,D] masked expansion followed by W_p and a
sum over neighbours, which counts b_p six times) so that quirks are reproduced, not re-derived.
"""
import numpy as np
import torch
import torch.nn.functional as F

T_STEPS = 4  # model.py:60

GGNN_KEYS = ["W_p", "W_z", "U_z", "W_r", "U_r", "W_h", "U_h"]


# --------------------------------------------------------------------------------------------------
# encoder index tables
def build_tables(roles_per_verb, verb_list, role_list):
    """imsitu_encoder.py:71-89 (roles_to_verb_tensor_list) and :158-159 (get_role_count).

    Returns (verb2roles int64 [V, R], role_count int64 [V]); pad value = len(role_list)."""
    max_role = max(len(roles_per_verb[v]) for v in verb_list)
    rid = {r: i for i, r in enumerate(role_list)}
    table = np.full((len(verb_list), max_role), len(role_list), dtype=np.int64)
    count = np.zeros(len(verb_list), dtype=np.int64)
    for vi, v in enumerate(verb_list):
        roles = roles_per_verb[v]
        count[vi] = len(roles)
        for k, r in enumerate(roles):
            table[vi, k] = rid[r]
    return table, count


def get_role_ids_batch(verb2roles, verbs):
    """imsitu_encoder.py:172-180: stack of verb2roles[verb] rows -> int64 [B, R]."""
    verbs = np.asarray(verbs, dtype=np.int64)
    return np.stack([verb2roles[int(v)] for v in verbs]) if len(verbs) else np.zeros((0, verb2roles.shape[1]), np.int64)


def get_adj_matrix_noself(role_count, verbs, max_role_count):
    """imsitu_encoder.py:209-229: outer product of the {1,0} role encoding, real diagonal zeroed, pad diagonal set."""
    verbs = np.asarray(verbs, dtype=np.int64)
    out = np.zeros((len(verbs), max_role_count, max_role_count), dtype=np.float32)
    for b, v in enumerate(verbs):
        n = int(role_count[int(v)])
        enc = np.zeros(max_role_count, dtype=np.int64)
        enc[:n] = 1                                   # verb2role_encoding, :93-112
        adj = np.outer(enc, enc)                      # expanded * transpose, :217-220
        for i in range(n):
            adj[i, i] = 0                             # :221-222
        for i in range(n, max_role_count):
            adj[i, i] = 1                             # :223-225
        out[b] = adj.astype(np.float32)               # :228 FloatTensor
    return out


# --------------------------------------------------------------------------------------------------
# GGSNN
def linear(x, w, b):
    return x @ w.t() + b


# The GRU's activations, looked up in this module at every call.  Tests rebind these names (never torch's own functions)
# to give the backward other derivative factors, e.g. to emulate the CUDA path's bf16 stash (tests/regimes.py).
gate_z = torch.sigmoid
gate_r = torch.sigmoid
candidate = torch.tanh


def ggsnn_forward(p, hidden_state, mask=None, verb=False, steps=T_STEPS, trace=None):
    """model.py:59-86.  p: dict with '<name>.weight' / '<name>.bias' for W_p,W_z,U_z,W_r,U_r,W_h,U_h."""
    for t in range(steps):
        if verb:
            neighbours = linear(hidden_state, p["W_p.weight"], p["W_p.bias"])            # :62-64
        else:
            batch_size, R = mask.shape[0], mask.shape[1]
            nb = hidden_state.contiguous().view(batch_size, R, -1)                      # :67-68
            nb = nb.expand(R, nb.size(0), nb.size(1), nb.size(2)).transpose(0, 1)       # :69-72
            nb = nb * mask.unsqueeze(-1)                                                # :73
            nb = linear(nb, p["W_p.weight"], p["W_p.bias"])                             # :74 (bias on all 6 neighbours)
            nb = torch.sum(nb, 2)                                                       # :75
            neighbours = nb.contiguous().view(batch_size * R, -1)                       # :76-77
        z_t = gate_z(linear(neighbours, p["W_z.weight"], p["W_z.bias"]) +
                     linear(hidden_state, p["U_z.weight"], p["U_z.bias"]))        # :80
        r_t = gate_r(linear(neighbours, p["W_r.weight"], p["W_r.bias"]) +
                     linear(hidden_state, p["U_r.weight"], p["U_r.bias"]))        # :81
        h_hat = candidate(linear(neighbours, p["W_h.weight"], p["W_h.bias"]) +
                          linear(r_t * hidden_state, p["U_h.weight"], p["U_h.bias"]))   # :82-83
        if trace is not None:
            trace.append({"m": neighbours, "z": z_t, "r": r_t, "h_hat": h_hat, "h_in": hidden_state})
        hidden_state = (1 - z_t) * hidden_state + z_t * h_hat                            # :84
    return hidden_state


def dropout(x, keep, p):
    """nn.Dropout(p) in training mode with an explicit Bernoulli keep-mask (model.py:106,110); identity if keep is None."""
    if keep is None or p == 0.0:
        return x
    return x * keep.to(x.dtype) / (1.0 - p)


# --------------------------------------------------------------------------------------------------
# FCGGNN stage (backbones bypassed: `feat` is what convnet_*(img) returns, [B, D])
def predict_nouns(params, feat, verbs, verb2roles, role_count, keep=None, drop_p=0.5):
    """model.py:114-155 with img_features := feat.  Runs on feat's device (fp64 on a GPU for the large cases)."""
    B = feat.shape[0]
    R = verb2roles.shape[1]
    verbs = verbs.to(feat.device)
    role_idx = torch.from_numpy(get_role_ids_batch(verb2roles, verbs.cpu().numpy())).to(feat.device)  # :117
    f = feat.expand(R, B, feat.size(1)).transpose(0, 1).contiguous().view(B * R, -1)     # :124-129
    verb_embd = params["verb_emb.weight"][verbs]                                         # :132
    role_embd = params["role_emb.weight"][role_idx].view(B * R, -1)                      # :133-135
    v = verb_embd.expand(R, B, verb_embd.size(1)).transpose(0, 1).contiguous().view(B * R, -1)  # :137-141
    node = F.relu(f * role_embd * v)                                                     # :143-144
    mask = torch.from_numpy(get_adj_matrix_noself(role_count, verbs.cpu().numpy(), R)).to(feat.device, feat.dtype)  # :147
    out = ggsnn_forward(_sub(params, "ggsnn."), node, mask=mask, verb=False)             # :151
    logits = linear(dropout(out, keep, drop_p), params["nouns_classifier.1.weight"],
                    params["nouns_classifier.1.bias"])                                   # :152
    return logits.contiguous().view(B, R, -1)                                            # :155


def predict_verb(params, feat, keep=None, drop_p=0.5):
    """model.py:157-168 with img_features := feat."""
    node = F.relu(feat)                                                                  # :160
    out = ggsnn_forward(_sub(params, "ggsnn."), node, mask=None, verb=True)              # :166
    return linear(dropout(out, keep, drop_p), params["verb_classifier.1.weight"],
                  params["verb_classifier.1.bias"])                                      # :168


def forward(params, feat_verbs, feat_nouns, gt_verb, verb2roles, role_count, keeps=(None, None, None), drop_p=0.5,
            pred_verbs=None):
    """model.py:171-180.  keeps = dropout keep-masks for (verb path, predicted-verb noun path, gt-verb noun path).

    pred_verbs (test infrastructure, not in the reference): verb ids to condition the predicted-verb noun path on
    instead of argmax(pred_verb).  With random-init weights the verb logits are nearly tied, so bf16 arithmetic flips
    ~1 % of the argmaxes; feeding the CUDA path's own predictions keeps the two role graphs identical and makes the
    pred-noun logits / gradients comparable row by row."""
    pred_verb = predict_verb(params, feat_verbs, keeps[0], drop_p)                       # :175
    verbs = torch.argmax(pred_verb, 1) if pred_verbs is None else pred_verbs
    pred_nouns = predict_nouns(params, feat_nouns, verbs, verb2roles, role_count,
                               keeps[1], drop_p)                                         # :176-177
    gt_pred_nouns = predict_nouns(params, feat_nouns, gt_verb, verb2roles, role_count, keeps[2], drop_p)  # :178
    return pred_verb, pred_nouns, gt_pred_nouns


def verb_loss(pred_verb, gt_verb):
    """model.py:182-187."""
    return F.cross_entropy(pred_verb, gt_verb)


def nouns_loss(pred_nouns, gt_nouns, num_labels):
    """model.py:189-201: sum over the 3 annotations of CE with ignore_index = num_labels (mean over non-ignored)."""
    loss = 0
    pn = pred_nouns.transpose(1, 2)                                                      # :195
    for i in range(3):
        loss = loss + F.cross_entropy(pn, gt_nouns[:, i], ignore_index=num_labels)       # :196-199
    return loss


def _sub(params, prefix):
    return {k[len(prefix):]: v for k, v in params.items() if k.startswith(prefix)}


# --------------------------------------------------------------------------------------------------
# parameters with the reference's default initialisation (nn.Linear: U(+-1/sqrt(fan_in)); nn.Embedding: N(0,1),
# padding row zero -- model.py:95-98,47-56,105-111), generated without importing the reference.
def init_params(num_verbs, num_roles, num_labels, D, seed=0, dtype=torch.float32):
    g = torch.Generator().manual_seed(seed)
    p = {}

    def lin(name, out_f, in_f):
        bound = 1.0 / (in_f ** 0.5)
        p[name + ".weight"] = ((torch.rand(out_f, in_f, generator=g) * 2 - 1) * bound).to(dtype)
        p[name + ".bias"] = ((torch.rand(out_f, generator=g) * 2 - 1) * bound).to(dtype)

    role = torch.randn(num_roles + 1, D, generator=g)
    role[num_roles] = 0
    p["role_emb.weight"] = role.to(dtype)
    p["verb_emb.weight"] = torch.randn(num_verbs, D, generator=g).to(dtype)
    for k in GGNN_KEYS:
        lin("ggsnn." + k, D, D)
    lin("verb_classifier.1", num_verbs, D)
    lin("nouns_classifier.1", num_labels, D)
    return p


def train_step_grads(params, feat_verbs, feat_nouns, gt_verb, gt_nouns, verb2roles, role_count, num_labels,
                     keeps=(None, None, None), drop_p=0.5, pred_verbs=None):
    """sr.py:63-79 without AMP: loss = verb_loss + nouns_loss(pred path); returns (losses, grads dict).
    gt_nouns_loss is computed but not back-propagated (sr.py:70,76)."""
    ps = {k: v.detach().clone().requires_grad_(True) for k, v in params.items()}
    pv, pn, gpn = forward(ps, feat_verbs, feat_nouns, gt_verb, verb2roles, role_count, keeps, drop_p, pred_verbs)
    vl = verb_loss(pv, gt_verb)
    nl = nouns_loss(pn, gt_nouns, num_labels)
    gl = nouns_loss(gpn, gt_nouns, num_labels)
    (vl + nl).backward()
    grads = {k: (v.grad if v.grad is not None else torch.zeros_like(v)) for k, v in ps.items()}
    return (vl.detach(), nl.detach(), gl.detach()), grads, (pv.detach(), pn.detach(), gpn.detach())


def train_step_grads_chunked(params, feat_verbs, feat_nouns, gt_verb, gt_nouns, verb2roles, role_count, num_labels,
                             keeps=(None, None, None), drop_p=0.5, pred_verbs=None, chunk=256, shard=None,
                             keep_logits=False):
    """The same step as train_step_grads on a batch too large for one pass of the as-written arithmetic (the
    [B,6,6,D] expansion of model.py:67-73 is 1.8 GB per copy at B = 6144): the batch is processed in chunks of `chunk`
    images with the GLOBAL loss denominators (B for the verb loss, the non-ignored target counts per annotation for
    the noun losses, model.py:184-185,196-199) and the gradients are summed, which is what one full-batch backward
    computes.  shard = (lo, hi) restricts the sums to that slice of the batch while keeping the global denominators
    (the per-rank share of a data-parallel step, sr.py:66-76 on GPU 0 of the reference's DataParallel)."""
    B = feat_verbs.shape[0]
    lo, hi = (0, B) if shard is None else shard
    counts = [(gt_nouns[:, a] != num_labels).sum().clamp_min(1).to(torch.float32) for a in range(3)]
    ps = {k: v.detach().clone().requires_grad_(True) for k, v in params.items()}
    tot = torch.zeros(3, dtype=torch.float64)
    logits = ([], [], [])
    for c0 in range(lo, hi, chunk):
        c1 = min(hi, c0 + chunk)
        sl = slice(c0, c1)
        kp = tuple(None if k is None else k[(c0 if i == 0 else c0 * verb2roles.shape[1]):
                                            (c1 if i == 0 else c1 * verb2roles.shape[1])] for i, k in enumerate(keeps))
        pvb = None if pred_verbs is None else pred_verbs[sl]
        pv, pn, gpn = forward(ps, feat_verbs[sl], feat_nouns[sl], gt_verb[sl], verb2roles, role_count, kp, drop_p, pvb)
        vl = F.cross_entropy(pv, gt_verb[sl], reduction="sum") / B
        nl, gl = 0, 0
        for a in range(3):
            nl = nl + F.cross_entropy(pn.transpose(1, 2), gt_nouns[sl, a], ignore_index=num_labels,
                                      reduction="sum") / counts[a]
            gl = gl + F.cross_entropy(gpn.transpose(1, 2), gt_nouns[sl, a], ignore_index=num_labels,
                                      reduction="sum") / counts[a]
        (vl + nl).backward()
        vl, nl, gl = vl.detach(), nl.detach(), gl.detach()
        tot += torch.tensor([vl.item(), nl.item(), gl.item()], dtype=torch.float64)
        if keep_logits:
            for dst, src in zip(logits, (pv, pn, gpn)):
                dst.append(src.detach())
    grads = {k: (v.grad if v.grad is not None else torch.zeros_like(v)) for k, v in ps.items()}
    outs = tuple(torch.cat(x) for x in logits) if keep_logits else None
    return tuple(tot.to(torch.float32)), grads, outs
