"""Generate the supervised-learning fixtures FROM THE REFERENCE'S OWN PYTHON (build container only: needs /root/reference;
GPU tests never run this file, they read what it wrote):   python tests/golden/make_sl_golden.py

Lines in OpenSpiel's bridge bidding text format (the input of sl.py:87-117) over the 1,000 real boards of
boards_wb5_1000.npz: the deal as 52 chance actions (card c dealt to seat k mod 4 from the dealer North at chance position
k, brl_b200/sl.py deal_owners), a random legal auction through the reference's BiddingPhase (make_golden.play_auction)
as 52 + action, then a dummy play tail of 52 card actions; passed-out deals are 56 ints with no tail (a few are forced).
For every (line, call position) the example the reference's make_dataset would yield -- observation of the player to act
by wb5/utils.convert_obs for dealer N and no vulnerability, the legal mask by convert_leagal_action_mask, and the call as
the label -- is frozen.  Output (committed, small): sl_golden.npz -- the lines as their ints (line_ints, split by
line_len; tests write them out as text), and per example line, position, label, obs_bits (little-endian packbits of the 480 bits), mask, and the expected
deal table (the boards' hands, no double-dummy results).
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

import make_golden as mg  # noqa: E402  (registers the import stubs and puts the reference on sys.path)

from brl_b200.deals import boards_from_json, pack_deal_table, unpack_deal_table  # noqa: E402


def main():
    import json
    with open(os.path.join(mg.REF, "wb5", "dataset_for_vs_wb5.json")) as fh:
        data = json.load(fh)
    table, _, _, _, _ = boards_from_json(data)
    owners, _ = unpack_deal_table(table)
    rng = np.random.default_rng(20261020)
    lines, rec = [], dict(line=[], position=[], label=[], obs_bits=[], mask=[])
    for i, board in enumerate(data["logs"]):
        # chance order: position k deals card chance[k] to seat k % 4 (dealer North)
        by_seat = [rng.permutation(np.flatnonzero(owners[i] == s)) for s in range(4)]
        chance = np.stack(by_seat, axis=1).reshape(-1)
        forced = [0, 0, 0, 0] if i % 100 == 0 else None
        bias = 0.0 if i % 4 == 0 else 0.62  # uniform random-legal auctions, and realistic pass-biased ones
        calls, obs_rows, mask_rows, _ = mg.play_auction(board, 0, 0, 0, rng, bias, forced=forced)
        toks = list(chance) + [52 + c for c in calls]
        if len(toks) != 56:
            toks += list(rng.permutation(52))
        lines.append(np.array(toks, np.int8))
        for p, (c, o, m) in enumerate(zip(calls, obs_rows, mask_rows)):
            rec["line"].append(i); rec["position"].append(p); rec["label"].append(c)
            rec["obs_bits"].append(o); rec["mask"].append(m)
    np.savez_compressed(
        os.path.join(HERE, "sl_golden.npz"), line_ints=np.concatenate(lines), line_len=np.array([len(x) for x in lines], np.int16),
        line=np.array(rec["line"], np.int32), position=np.array(rec["position"], np.int32),
        label=np.array(rec["label"], np.int32), obs_bits=np.stack(rec["obs_bits"]).astype(np.uint8),
        mask=np.stack(rec["mask"]).astype(np.uint8), table=pack_deal_table(owners, np.zeros((len(owners), 4, 5), np.int64)))
    print(f"wrote {len(lines)} lines, {len(rec['line'])} examples")


if __name__ == "__main__":
    main()
