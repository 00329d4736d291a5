"""Timings of hand reading (DESIGN.md f18, f19) on self-play auctions of two seeded nets.

    python scripts/hand_reading_bench.py [out=profiles/r22_posterior_b200.json] [runs=5] [boards=100,1000] [samples=1024,4096]
        [legs=is,smc] [smc_out=profiles/r23_smc_b200.json]

For each board count: the auction-recording match (host match loop with record=), then posterior.hand_posterior over both
tables x 4 observers at the end of each auction, for each N and precision: median and range of `runs` calls (host clock
around a call that ends in a device synchronise), forward rows and rows/s.  A separate torch.profiler run at 1,000 boards and
N = 1,024 gives the share of the call's device time outside the grouped forward's kernels.  ESS median and 10th percentile at
temperature 1 and 0.  The card's name, power limit and max SM clock are read in the same run.

The SMC leg (legs=smc) reads 1,000 boards, both tables x 4 observers at the end of the auction, on two deal sets (the
synthetic table and the real boards of tests/golden/boards_wb5_1000.npz), at temperatures 1, 0.25 (standing in for a
sharper, trained net) and 0: SMC at N = 1,024 with R = 1 and R = 4 (kappa = 0.5), IS at N = 1,024 and IS at the N (a
multiple of 1,024) whose forward rows come closest to the SMC call's.  Per case: median time of `runs` calls, forward rows
(SMC: the reweights' rows plus an upper bound of the moves' rows, from the resample count and the most rows a pair can
need), ESS quantiles, the empty-query share, cards read and partner cards read (posterior.reading_stats) and the mean
acceptance."""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

DEFAULTS = dict(out="profiles/r22_posterior_b200.json", runs=5, boards="100,1000", samples="1024,4096", seed=0, legs="is,smc",
                smc_out="profiles/r23_smc_b200.json")


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as exc:  # noqa: BLE001
        q = f"unavailable ({exc})"
    return dict(nvidia_smi=q, torch_name=torch.cuda.get_device_name(0))


def main(argv):
    cfg = dict(DEFAULTS)
    for a in argv:
        k, _, v = a.partition("=")
        cfg[k] = type(DEFAULTS[k])(v)
    from brl_b200 import posterior
    from brl_b200.deals import synthetic_deal_table
    from tests.helpers import seeded_params
    dev = "cuda"
    if not torch.cuda.is_available():
        raise SystemExit("hand_reading_bench needs a GPU")
    nets = [seeded_params(1, dev), seeded_params(2, dev)]
    table = synthetic_deal_table(1000, seed=0)
    if "smc" in cfg["legs"].split(","):
        smc_leg(cfg, nets, table)
    if "is" not in cfg["legs"].split(","):
        return
    result = dict(gpu=gpu_info(), runs=cfg["runs"], note="ESS on trained nets has not been measured; these are seeded nets",
                  cases=[])
    for boards in [int(x) for x in cfg["boards"].split(",")]:
        t0 = time.perf_counter()
        rec = posterior.selfplay_auctions(nets[0], nets[1], table, boards, seed=cfg["seed"], device=dev)
        torch.cuda.synchronize()
        record_s = time.perf_counter() - t0
        queries, seat_nets = posterior.reading_queries(rec["offsets"], rec["seat_nets"], rec["dealer"], "end")
        segs = posterior.query_segments(queries, seat_nets, rec["dealer"][queries[:, 0]])
        calls_read = sum(sum(s.values()) for s in segs)
        for N in [int(x) for x in cfg["samples"].split(",")]:
            for precision in (None, "tc-bf16"):
                kw = dict(board=rec["board"], dealer=rec["dealer"], vul=rec["vul"], samples=N, seed=1, precision=precision)
                times = []
                post = None
                for r in range(cfg["runs"] + 1):  # the first call warms up
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    post = posterior.hand_posterior(nets, table, rec["calls"], rec["offsets"], queries, seat_nets, **kw)
                    torch.cuda.synchronize()
                    if r:
                        times.append(time.perf_counter() - t0)
                zero = posterior.hand_posterior(nets, table, rec["calls"], rec["offsets"], queries, seat_nets, temperature=0.0, **kw)
                ess = lambda p: [float(np.nanmedian(p["ess"])), float(np.nanpercentile(p["ess"], 10)),  # noqa: E731
                                 float((p["accepted"] == 0).mean())]
                rows = calls_read * N
                case = dict(boards=boards, queries=int(queries.shape[0]), samples=N, precision=precision or "tc",
                            record_match_s=record_s, call_s_median=float(np.median(times)), call_s_range=[min(times), max(times)],
                            forward_rows=rows, rows_per_s=rows / float(np.median(times)),
                            ess_tau1_median_p10_noaccept=ess(post), ess_tau0_median_p10_noaccept=ess(zero))
                print(json.dumps(case), flush=True)
                result["cases"].append(case)
    # the share outside the grouped forward, in a profiler run of its own
    rec = posterior.selfplay_auctions(nets[0], nets[1], table, 1000, seed=cfg["seed"], device=dev)
    queries, seat_nets = posterior.reading_queries(rec["offsets"], rec["seat_nets"], rec["dealer"], "end")
    kw = dict(board=rec["board"], dealer=rec["dealer"], vul=rec["vul"], samples=1024, seed=1)
    posterior.hand_posterior(nets, table, rec["calls"], rec["offsets"], queries, seat_nets, **kw)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        posterior.hand_posterior(nets, table, rec["calls"], rec["offsets"], queries, seat_nets, **kw)
        torch.cuda.synchronize()
    by = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
        if t:
            by[e.key] = by.get(e.key, 0) + t
    post_k = {k: v for k, v in by.items() if "k_post_" in k}
    other_k = {k: v for k, v in by.items() if "k_post_" not in k}
    total = sum(by.values())
    result["profile_1000_boards_N1024"] = dict(
        device_us_total=total, posterior_kernels_us=post_k, share_outside_forward=sum(post_k.values()) / total if total else None,
        forward_and_copies_us=sum(other_k.values()), top_other=sorted(other_k.items(), key=lambda kv: -kv[1])[:8])
    print(json.dumps(result["profile_1000_boards_N1024"]), flush=True)
    os.makedirs(os.path.dirname(cfg["out"]) or ".", exist_ok=True)
    with open(cfg["out"], "w") as fh:
        json.dump(result, fh, indent=1)


def _timed(fn, runs):
    times, out = [], None
    for r in range(runs + 1):  # the first call warms up
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        if r:
            times.append(time.perf_counter() - t0)
    return out, times


def _smc_move_rows_bound(post, queries, seat_nets, dealers, N, moves):
    """an upper bound of the rows the moves ran: per query, resamples x R x N x the most calls a pair held at any stage"""
    from brl_b200 import posterior
    segs = posterior.smc_segments(queries, seat_nets, dealers, True)
    most = np.array([max((sum(v.values()) for key, v in sg.items() if key[0] == "m"), default=0) for sg in segs])
    return int((post["resamples"].astype(np.int64) * moves * N * most).sum())


def smc_leg(cfg, nets, synthetic):
    from brl_b200 import posterior
    from brl_b200.deals import unpack_deal_table
    from tests.helpers import load_boards
    result = dict(gpu=gpu_info(), runs=cfg["runs"], kappa=0.5,
                  note="seeded (untrained) nets; temperature 0.25 stands in for a sharper net; trained nets not measured",
                  cases=[])
    real = load_boards()["table"]
    N = 1024
    for deals_name, table in (("synthetic", synthetic), ("boards_wb5_1000", real)):
        rec = posterior.selfplay_auctions(nets[0], nets[1], table, 1000, seed=cfg["seed"], device="cuda")
        queries, seat_nets = posterior.reading_queries(rec["offsets"], rec["seat_nets"], rec["dealer"], "end")
        dealers = rec["dealer"][queries[:, 0]].astype(np.int64)
        calls_read = sum(sum(s.values()) for s in posterior.query_segments(queries, seat_nets, dealers))
        owners, _ = unpack_deal_table(table)
        base = dict(board=rec["board"], dealer=rec["dealer"], vul=rec["vul"], seed=1)
        for tau in (1.0, 0.25, 0.0):
            def case(label, post, times, rows, **extra):
                stats = posterior.reading_stats(post, queries, seat_nets, owners, rec["board"])
                ess = post["ess"][post["accepted"] > 0]
                c = dict(deals=deals_name, temperature=tau, method=label, queries=int(queries.shape[0]),
                         call_s_median=float(np.median(times)), call_s_range=[min(times), max(times)], forward_rows=rows,
                         ess_p10_p50_p90=[float(np.percentile(ess, q)) for q in (10, 50, 90)] if ess.size else None,
                         empty_share=float((post["accepted"] == 0).mean()),
                         cards_read=float(np.mean([v["cards_read"] for v in stats.values() if v["cards_read"] is not None])),
                         partner_cards_read=float(np.mean([v["partner_cards_read"] for v in stats.values()
                                                           if v["partner_cards_read"] is not None])), **extra)
                print(json.dumps(c), flush=True)
                result["cases"].append(c)
                return c
            smc_rows = []
            for R in (1, 4):
                post, times = _timed(lambda: posterior.hand_posterior(nets, table, rec["calls"], rec["offsets"], queries, seat_nets,
                                                                      samples=N, temperature=tau, method="smc", moves=R,
                                                                      ess_threshold=0.5, **base), cfg["runs"])
                rows = calls_read * N + _smc_move_rows_bound(post, queries, seat_nets, dealers, N, R)
                smc_rows.append(rows)
                acc = post["acceptance"][np.isfinite(post["acceptance"])]
                case(f"smc R={R}", post, times, rows, samples=N, moves=R, forward_rows_is_upper_bound=True,
                     resamples_mean=float(post["resamples"].mean()), acceptance_mean=float(acc.mean()) if acc.size else None)
            for n_is in sorted({N} | {N * max(1, int(round(r / (calls_read * N)))) for r in smc_rows}):
                post, times = _timed(lambda: posterior.hand_posterior(nets, table, rec["calls"], rec["offsets"], queries, seat_nets,
                                                                      samples=n_is, temperature=tau, **base), cfg["runs"])
                case("is", post, times, calls_read * n_is, samples=n_is)
    os.makedirs(os.path.dirname(cfg["smc_out"]) or ".", exist_ok=True)
    with open(cfg["smc_out"], "w") as fh:
        json.dump(result, fh, indent=1)


if __name__ == "__main__":
    main(sys.argv[1:])
