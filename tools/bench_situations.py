"""Top-k situation decode on one GPU: FCGGNN.situations_from_features at D = 2048 on the synthetic 504 / 190 / 2001
vocabulary with imSitu's role histogram, B in {768, 6144} x k in {1, 5}, eager and replayed from a CUDA graph.

Per configuration: ms per call, images/s and situations/s; the same run also times the verb path alone and one k = 1
role-graph pass (the bar: a k-candidate call against the verb path + k single-candidate passes), the row kernel
`k_row_topk_logsoftmax` on the noun logits by CUDA events (achieved GB/s on its algorithmic bytes, against the
6550 GB/s copy bandwidth DESIGN.md uses), and the GEMMs' TFLOP/s from the library's per-GEMM event bracket
(srg_profile_*).  The card's name, power limit and SM clock are read in the same run.  Prints one JSON line."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import situation_recognition_b200 as S  # noqa: E402
from situation_recognition_b200 import _lib  # noqa: E402
from situation_recognition_b200.synthetic import make_batch, make_train_json  # noqa: E402
from bench import ClockSampler  # noqa: E402

COPY_GBPS = 6550.0     # measured device copy bandwidth of a B200 (DESIGN.md section 4.2)


def card_info():
    out = {"name": torch.cuda.get_device_name(), "power_limit_w": None}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        out["power_limit_w"] = float(q.strip().splitlines()[0])
    except Exception:
        pass
    return out


def timed(fn, iters):
    """ms per call: CUDA events around `iters` back-to-back calls."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def preheat(fn, seconds):
    t0 = time.perf_counter()
    n = 0
    while time.perf_counter() - t0 < seconds:
        fn()
        n += 1
        if n % 8 == 0:
            torch.cuda.synchronize()
    torch.cuda.synchronize()


def graphed(fn):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    return g


def gemm_tflops(lib, fn):
    kinds = 32
    ms, fl, ct = (ctypes.c_double * kinds)(), (ctypes.c_double * kinds)(), (ctypes.c_longlong * kinds)()
    lib.srg_profile_begin()
    fn()
    _lib.check(lib.srg_profile_end(kinds, ms, fl, ct))
    tms, tfl = sum(ms), sum(fl)
    return {"gemm_ms": tms, "gemm_tflops": tfl / max(tms, 1e-9) / 1e9, "gemm_launches": int(sum(ct))}


def topk_kernel(lib, rows, n, ldl, k, iters):
    """Event-timed srg_topk_logsoftmax on a [rows, ldl] fp32 buffer (first n columns); two buffers alternate so that
    a working set above the 126 MB L2 is read from HBM."""
    bufs = [torch.randn(rows, ldl, device="cuda") for _ in range(2)]
    idx = torch.empty(rows, k, dtype=torch.int64, device="cuda")
    lp = torch.empty(rows, k, dtype=torch.float32, device="cuda")
    st = _lib.stream_ptr()
    calls = [lambda x=x: _lib.check(lib.srg_topk_logsoftmax(_lib.ptr(x), ldl, rows, n, k, _lib.ptr(idx),
                                                             _lib.ptr(lp), st)) for x in bufs]
    step = lambda: (calls[0](), calls[1]())   # noqa: E731
    step()
    ms = timed(step, iters) / 2
    nbytes = rows * n * 4 + rows * k * 12
    return {"rows": rows, "n": n, "k": k, "ms": ms, "gb_per_s": nbytes / ms / 1e6,
            "of_copy_bw": nbytes / ms / 1e6 / COPY_GBPS, "l2_resident": 2 * rows * ldl * 4 < 126e6}


def main():
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--D", type=int, default=2048)
    ap.add_argument("--batches", default="768,6144")
    ap.add_argument("--ks", default="1,5")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--preheat", type=float, default=3.0, help="seconds of untimed calls before each timed region")
    ap.add_argument("--out", default="", help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_situations.py needs a B200: the decode has no CPU path")
    torch.manual_seed(0)
    enc = S.imsitu_encoder(make_train_json(seed=0), verbose=False)
    m = S.FCGGNN(enc, args.D, backbone=None, precision="bf16").cuda().eval()
    lib = _lib.load()
    R, L = enc.get_max_role_count(), enc.get_num_labels()
    Lpad = (L + 255) // 256 * 256
    clocks = ClockSampler(torch.cuda.current_device())
    clocks.start()
    results = []
    for B in [int(x) for x in args.batches.split(",")]:
        fv, fn, _, _ = make_batch(enc, B, args.D, seed=1234, device="cuda")
        with torch.no_grad():
            top = m.situations_from_features(fv, fn, k=max(int(x) for x in args.ks.split(","))).verbs
        verb_path = torch.no_grad()(lambda: m.predict_verb(fv, B))                         # eval, no autograd
        one = top[:, :1].contiguous()
        rg1 = lambda: m.situations_from_features(None, fn, verbs=one)                      # noqa: E731
        preheat(rg1, args.preheat)
        t_verb, t_rg1 = timed(verb_path, args.iters), timed(rg1, args.iters)
        for k in [int(x) for x in args.ks.split(",")]:
            call = lambda: m.situations_from_features(fv, fn, k=k)                       # noqa: E731
            preheat(call, args.preheat)
            eager = timed(call, args.iters)
            g = graphed(call)
            preheat(g.replay, args.preheat)
            graph = timed(g.replay, args.iters)
            del g
            best = min(eager, graph)
            res = {"B": B, "k": k, "ms_eager": eager, "ms_graph": graph,
                   "images_per_s": B / best * 1e3, "situations_per_s": B * k / best * 1e3,
                   "ms_verb_path": t_verb, "ms_role_graph_k1": t_rg1,
                   "vs_verb_plus_k_passes": eager / (t_verb + k * t_rg1),
                   "topk_nouns": topk_kernel(lib, B * k * R, L, Lpad, 1, args.iters),
                   "topk_verbs": topk_kernel(lib, B, enc.get_num_verbs(), 512, k, args.iters)}
            res.update(gemm_tflops(lib, call))
            results.append(res)
            torch.cuda.empty_cache()
    clk = clocks.stop()
    line = {"metric": "situations_decode", "D": args.D, "precision": "bf16", "card": card_info(), "clocks": clk,
            "preheat_s": args.preheat, "iters": args.iters, "results": results}
    s = json.dumps(line)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
