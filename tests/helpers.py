"""Shared test helpers: golden fixtures (made by tests/golden/make_golden.py from
the reference's own Python) and seeded episode draws."""
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# the 8 valid seatings: one team on N/S, the other on E/W (SURVEY A.1)
SEATINGS = np.array([[0, 2, 1, 3], [2, 0, 3, 1], [1, 2, 0, 3], [3, 0, 2, 1],
                     [0, 3, 1, 2], [2, 1, 3, 0], [1, 3, 0, 2], [3, 1, 2, 0]], dtype=np.int8)


def load_boards():
    z = np.load(os.path.join(GOLDEN, "boards_wb5_1000.npz"))
    return {k: z[k] for k in z.files}


def load_c1():
    """configs[0] golden match (tests/golden/make_c1_golden.py)"""
    z = np.load(os.path.join(GOLDEN, "c1_eval_match.npz"))
    return {k: z[k] for k in z.files}


def load_c1_seeded():
    """the configs[0] match played by two seeded nets (tests/golden/make_c1_golden.py --seeded)"""
    z = np.load(os.path.join(GOLDEN, "c1_seeded_match.npz"))
    return {k: z[k] for k in z.files}


def seeded_params(seed, device):
    """A net of the bundled models' architecture from a seed: haiku's initialisation (models.init_params) with the policy
    head scaled by 128 (exact in fp32), so that its logits have a trained net's magnitude and the top-2 gaps of a match
    stay far above the forward's rounding error."""
    from brl_b200.models import LAYERS, init_params
    p = init_params(seed, device)
    p[LAYERS[4]]["w"] *= 128
    return p


def weight_path(name):
    """bundled model pickle (bridge_models/ of the reference, 15 MB each): not in the repository; copy it to
    tests/golden/_weights/ (git-ignored) to run the checks that use it"""
    path = os.path.join(GOLDEN, "_weights", name)
    if not os.path.exists(path):
        raise FileNotFoundError(f"{path} is missing")
    return path


def load_auctions():
    z = np.load(os.path.join(GOLDEN, "auctions.npz"))
    return {k: z[k] for k in z.files}


def load_known():
    with open(os.path.join(GOLDEN, "known_auctions.json")) as fh:
        return json.load(fh)


def unpack_obs_bits(bits):
    """u8[...,60] little-endian packed -> u8[...,480]"""
    return np.unpackbits(np.asarray(bits, dtype=np.uint8), axis=-1, bitorder="little")[..., :480]


def auction_matrix(gold):
    """calls as a dense [A, Lmax] matrix padded with -1, plus lengths."""
    off = gold["offsets"]
    lens = np.diff(off)
    a = len(lens)
    mat = np.full((a, int(lens.max())), -1, dtype=np.int32)
    for i in range(a):
        mat[i, : lens[i]] = gold["calls"][off[i]: off[i + 1]]
    return mat, lens


def expected_rewards(final_row, players):
    """rewards by player id: + declarer-score for the declaring team, - for the other."""
    decl, _, _, _, _, sc = [int(v) for v in final_row]
    if decl < 0:
        return np.zeros(4, np.float32)
    team = int(players[decl]) // 2
    return np.array([sc if (pid // 2) == team else -sc for pid in range(4)], np.float32)
