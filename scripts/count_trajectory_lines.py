"""How compressible is bench.py's trajectory?  Counts, on the CPU oracle, the 32-byte sectors and 128-byte lines of the
[32, 8192, 480] f32 observation and [32, 8192, 38] u8 mask trajectories that are entirely zero, and the lines that hold one
repeated non-zero 32-bit value.  Same deal table, keys and Philox action stream as bench.py (launch i covers steps
32 i .. 32 i + 31); launch 0 starts from freshly dealt boards, later launches are the steady state the bench times.

    python scripts/count_trajectory_lines.py [launches]   # prints one JSON line per launch counted
"""
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from brl_b200.deals import synthetic_deal_table  # noqa: E402
from oracle import oracle as orc  # noqa: E402

N_ENVS, T_STEPS, N_DEALS, SEED = 8192, 32, 100_000, 20241017  # bench.py


def line_counts(buf: np.ndarray) -> dict:
    b = np.frombuffer(buf.tobytes(), dtype=np.uint8)
    b = np.concatenate([b, np.zeros((-len(b)) % 128, np.uint8)])  # the allocation's tail is a whole line
    sectors = b.reshape(-1, 32)
    lines = b.reshape(-1, 128)
    words = lines.view(np.uint32)
    zero_lines = ~lines.any(axis=1)
    uniform = (words == words[:, :1]).all(axis=1)
    return {"bytes": int(buf.nbytes), "sectors": len(sectors), "zero_sectors": int((~sectors.any(axis=1)).sum()),
            "lines": len(lines), "zero_lines": int(zero_lines.sum()), "uniform_nonzero_lines": int((uniform & ~zero_lines).sum()),
            "zero_line_frac": round(float(zero_lines.mean()), 4), "zero_sector_frac": round(float((~sectors.any(axis=1)).mean()), 4)}


def main():
    launches = int(sys.argv[1]) if len(sys.argv) > 1 else 5
    env = orc.OracleEnv(synthetic_deal_table(N_DEALS, seed=0), N_ENVS, n_threads=os.cpu_count() or 1)
    env.init(orc.make_keys(SEED, N_ENVS))
    for i in range(launches):
        out = env.rollout_random(SEED, i * T_STEPS, T_STEPS)
        if i == 0 or i == launches - 1:
            print(json.dumps({"launch": i, "steps": [i * T_STEPS, (i + 1) * T_STEPS - 1],
                              "observation_f32": line_counts(out["observation"]),
                              "legal_action_mask_u8": line_counts(out["legal_action_mask"])}))


if __name__ == "__main__":
    main()
