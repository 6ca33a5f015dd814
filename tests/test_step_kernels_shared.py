"""The virtual-loss step kernel (AZ_F_VIRTUAL_LOSS) starts a search and expands its root with the exact kernel's code: its root
requests are reported like the exact kernel's, and its noisy root priors are the exact kernel's bit for bit."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

N_TREES, K, SEED = 256, 4, 5


def _engine(leaves, n_playouts):
    from alphazero_openspiel_b200 import engine as E, _lib as L
    flags = L.F_KEEP_TREE | L.F_SAMPLE_MOVES | (L.F_VIRTUAL_LOSS if leaves else 0)
    return E.Engine("connect_four", N_TREES, n_playouts=n_playouts, noise_mode=L.NOISE_COUNTER, eval_mode=L.EVAL_HASH,
                    flags=flags, seed=SEED, leaves_per_tree=max(leaves, 1))


def test_virtual_loss_root_request_reports_the_root():
    """A tree waiting for the evaluation of a later move's root reports that root: az_request_info gives the root's position
    and az_status the root's legal-move count (not those of the tree's last leaf request)."""
    from alphazero_openspiel_b200 import _lib as L
    eng = _engine(K, n_playouts=16)
    checked = 0
    for _ in range(200):
        eng.step()
        st = eng.status()
        pos = eng.positions()
        sel = np.nonzero((st["phase"] == L.PH_ROOT_EVAL) & (pos["ply"] >= 1))[0]
        if len(sel) == 0:
            continue
        info = eng.request_info(max_depth=1)
        assert np.array_equal(info["bb"][sel], pos["bb"][sel])
        assert np.array_equal(info["ply"][sel], pos["ply"][sel])
        assert np.all(info["depth"][sel] == 0)
        occ = pos["bb"][sel, 0] | pos["bb"][sel, 1]
        n_legal = [bin(int(~int(o) >> 35) & 0x7F).count("1") for o in occ]   # Connect Four: columns whose top cell is empty
        assert list(st["req_legal"][sel]) == n_legal
        checked += len(sel)
        if checked >= N_TREES:
            break
    eng.close()
    assert checked >= N_TREES


def test_virtual_loss_root_priors_are_the_exact_kernels():
    """AZ_NOISE_COUNTER root expansion: the noisy priors of the first root are the exact kernel's, bit for bit."""
    from alphazero_openspiel_b200 import _lib as L
    child_p = {}
    for leaves in (0, K):
        eng = _engine(leaves, n_playouts=100)
        eng.step()   # root requests
        assert np.all(eng.phases().cpu().numpy() == L.PH_ROOT_EVAL)
        eng.step()   # root expansion, then the first simulations
        rs = eng.root_stats(offpolicy=False)
        assert np.all(rs["n_children"] == 7) and np.all(eng.positions()["ply"] == 0)
        child_p[leaves] = rs["child_p"]
        eng.close()
    assert np.array_equal(child_p[0].view(np.uint64), child_p[K].view(np.uint64))
