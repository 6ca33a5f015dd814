"""Generates the Breakthrough 6x6 fixtures by running the UNMODIFIED reference network (network.py of a checkout of
danielwillemsen/alphazero-openspiel) with its shipped checkpoint:

    python tests/golden/make_golden_bt6.py REFERENCE_CHECKOUT

  example_model_breakthrough_6x6.pth  the reference's models/example_model_breakthrough(6x6).pth (weights are data;
                                      BASELINE config [1] runs "with the shipped model", which cannot travel otherwise)
  bt6_pins.npz                        64 random non-terminal positions (action histories), reference Net priors [64,432]
                                      and values [64] in fp32, and the legal-move lists -- the pins of the observation /
                                      action encoding for Breakthrough and of the evaluator kernels' numerics.
"""
import os
import shutil
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import pyspiel_shim  # noqa: E402

pyspiel = pyspiel_shim.install()
REF = os.path.abspath(sys.argv[1])
sys.path.insert(0, REF)
import torch  # noqa: E402
import network as ref_network  # noqa: E402

if __name__ == "__main__":
    ck = os.path.join(REF, "models", "example_model_breakthrough(6x6).pth")
    shutil.copyfile(ck, os.path.join(HERE, "example_model_breakthrough_6x6.pth"))
    game = "breakthrough(rows=6,columns=6)"
    g = pyspiel.load_game(game)
    net = ref_network.Net([3, 6, 6], 432)
    net.load_state_dict(torch.load(ck, map_location="cpu", weights_only=True))
    net.eval()
    rng = np.random.RandomState(6)
    hists, boards, legal = [], [], []
    while len(hists) < 64:
        s = g.new_initial_state()
        for _ in range(rng.randint(0, 40)):
            if s.is_terminal():
                break
            s.apply_action(int(rng.choice(s.legal_actions())))
        if s.is_terminal():
            continue
        hists.append(s.history())
        boards.append(ref_network.state_to_board(s, [3, 6, 6]))
        legal.append(s.legal_actions())
    with torch.no_grad():
        p, v = net(torch.from_numpy(np.array(boards)).float())
    H = np.full((64, 40), -1, dtype=np.int32)
    for i, h in enumerate(hists):
        H[i, :len(h)] = h
    Lg = np.full((64, 48), -1, dtype=np.int32)
    for i, l in enumerate(legal):
        Lg[i, :len(l)] = l
    np.savez_compressed(os.path.join(HERE, "bt6_pins.npz"), histories=H, p=p.numpy().astype(np.float32),
                        v=v.numpy()[:, 0].astype(np.float32), legal=Lg)
    mass = [float(p[i, legal[i]].sum()) for i in range(64)]
    print("wrote bt6_pins.npz; mean policy mass on legal moves %.4f" % np.mean(mass))
