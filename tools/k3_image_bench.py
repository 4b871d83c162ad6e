"""k_constraints input traffic and timing at the bench shape (1 024 random worlds x 10 obstacles, Kinova, 128 steps).

Reports, from the counts of the built batch, the bytes one launch must fetch in 32-byte sectors and 128-byte lines under
  * the padded layout (tables at capL / capU strides, candidate records level-major [chunk][level][row]), and
  * the packed evaluation images (one contiguous run per chunk),
next to CUDA-event timings of eval_device (g + dense Jacobian of every world per launch).

    python tools/k3_image_bench.py [--worlds 1024] [--obstacles 10] [--launches 50] [--out FILE.json]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
NF = 7


def touched(start, length, unit):
    """units of `unit` bytes covering [start, start + length) (0 when length is 0), element-wise"""
    start, length = np.asarray(start, np.int64), np.asarray(length, np.int64)
    return np.where(length > 0, (start + length - 1) // unit - start // unit + 1, 0)


def padded_bytes(ln, un, cnt, capL, capU, T, NJ, O, TB, unit):
    """bytes one launch fetches from the padded tables and the level-major candidate records"""
    P = ln.shape[0]
    lt = np.arange(P * T * NJ, dtype=np.int64)
    n = ln.reshape(-1).astype(np.int64)
    b = touched(lt * capL * 2, n * 2, unit).sum() + touched(lt * capL * 24, n * 24, unit).sum()
    ut = np.arange(P * T * NF, dtype=np.int64)
    n = un.reshape(-1).astype(np.int64)
    b += touched(ut * capU * 2, n * 2, unit).sum() + touched(ut * capU * 8, n * 8, unit).sum()
    # centres, radii, counts: contiguous per chunk
    nch = P * (T // TB)
    b += nch * (2 * touched(0, TB * NJ * 24, unit) + 2 * touched(0, TB * NF * 8, unit) + touched(0, TB * NF * 4, unit)
                + touched(0, TB * NJ * 4, unit) + touched(0, TB * NJ * O, unit))
    # candidate records: [chunk][level][row], 32 B each
    rows = NJ * TB * O
    c = cnt.reshape(nch, rows).astype(np.int64)
    c = np.where(c == 255, 0, c)
    lines = set()
    for q in range(int(c.max(initial=0))):
        ch, x = np.nonzero(c > q)
        lines.update(((ch * 32 * rows + q * rows + x) * 32 // unit).tolist())
    return (int(b) + len(lines)) * unit


def image_bytes(ln, un, cnt, T, NJ, O, TB, layout, unit):
    """bytes one launch fetches from the packed images: the header, then records and tables as one run"""
    P = ln.shape[0]
    nch = P * (T // TB)
    rows = NJ * TB * O
    c = cnt.reshape(nch, rows).astype(np.int64)
    stored = np.where(c == 255, 0, c).sum(axis=1)
    nl = ln.reshape(nch, TB * NJ).sum(axis=1).astype(np.int64)
    nu = un.reshape(nch, TB * NF).sum(axis=1).astype(np.int64)
    head = touched(0, layout["counts"] + rows, unit)
    body = touched(layout["records"], stored * 32 + nl * 32 + nu * 10, unit)
    return int((head + body).sum() * unit)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worlds", type=int, default=1024)
    ap.add_argument("--obstacles", type=int, default=10)
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--seed", type=int, default=20261017)
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    from armour_b200 import ReachSetEngine, worlds
    if not torch.cuda.is_available():
        raise SystemExit("k3_image_bench: no CUDA device")
    P, O = args.worlds, args.obstacles
    q0, qd0, qdd0, q_des, obs = worlds.random_problems(P, O, seed=args.seed)
    eng = ReachSetEngine(max_problems=P, max_obstacles=O)
    eng.build(q0, qd0, qdd0, obs)
    T, NJ, TB = eng.T, eng.NJ, eng.lib.armour_chunk_intervals()
    ln, un = eng.monomial_counts()
    cnt = eng.candidate_counts()
    layout = eng.eval_image_layout()
    capL, capU = eng.cfg.cap_link_monomials, eng.cfg.cap_torque_monomials
    res = {"worlds": P, "obstacles": O, "image_bytes_per_chunk_slot": layout["chunk"],
           "image_slot_bytes_per_world": layout["chunk"] * (T // TB)}
    for unit in (32, 128):
        res[f"padded_read_bytes_{unit}B"] = padded_bytes(ln, un, cnt, capL, capU, T, NJ, O, TB, unit)
        res[f"image_read_bytes_{unit}B"] = image_bytes(ln, un, cnt, T, NJ, O, TB, layout, unit)
    dev = torch.device("cuda")
    eng.set_stream(torch.cuda.current_stream().cuda_stream)  # the events below time this stream
    rng = np.random.default_rng(1)
    kk = [torch.tensor(rng.uniform(-1, 1, (P, NF)), dtype=torch.float64, device=dev) for _ in range(16)]
    m = eng.m
    g = torch.empty((P, m), dtype=torch.float64, device=dev)
    jac = torch.empty((P, m, NF), dtype=torch.float64, device=dev)
    for i in range(5):
        eng.eval_device(P, kk[i % 16].data_ptr(), g.data_ptr(), jac.data_ptr())
    torch.cuda.synchronize()
    times = []
    for rep in range(5):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(args.launches):
            eng.eval_device(P, kk[i % 16].data_ptr(), g.data_ptr(), jac.data_ptr())
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b) * 1e3 / args.launches)
    res["eval_device_us_per_launch"] = sorted(times)
    res["gpu"] = torch.cuda.get_device_name(0)
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
