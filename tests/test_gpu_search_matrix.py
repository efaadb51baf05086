"""The search kernels against the oracle on every dispatch instance (run with -m gpu on the B200 box).

engine.cu picks a different template instance of the select, noise, plan and expand + back-up kernels from the action
count and the minibatch's batch.  tests/search_matrix.py lists the cases and which instance each one reaches;
tests/test_host_search_matrix.py proves (without a GPU) that together they reach every instance.  Each case here is the
bit-exact parity of tests/test_gpu_parity.py: trees, float64 policies, Q, sampled moves, roots and status."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from harness import diff_tree, np_choice
from search_matrix import CHAIN_CASES, NOISE_BOARDS, PARITY_CASES, STUBS, VL_CASES, host_noise, make_roots, make_tree

pytestmark = pytest.mark.gpu

KIND_TERMINAL = 1  # csrc/engine.cuh


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def run_case(torch, case):
    """run_search_parity (tests/test_gpu_parity.py) generalised: `batch` may be below `max_batch`, the noise is either
    injected host Dirichlet draws or the device's Philox stream (captured through noise_out and replayed to the oracle),
    the network is the hash or the chain stub, and the engine may run virtual loss (the oracle then restates
    select_vl_kernel).  Returns the number of terminal descents and the longest descent path the engine recorded."""
    from caro_ai_b200.engine import SelfPlayEngine
    game = case.product_game()
    og = case.oracle_game()
    G, A, batch, tpg = case.G, case.A, case.batch, case.trees_per_game
    rng = np.random.default_rng(case.seed)
    roots = make_roots(case, og, rng)
    eng = SelfPlayEngine(game, G, trees_per_game=tpg, max_batch=case.max_batch,
                         node_capacity=case.count * batch * case.moves + 8, seed=case.seed, virtual_loss=case.virtual_loss)
    eng.set_roots([r[0] for r in roots], [r[1] for r in roots])
    trees = [[make_tree(case, og) for _ in range(tpg)] for _ in range(G)]
    stub = STUBS[case.stub]
    states = [r[0] for r in roots]
    players = [r[1] for r in roots]
    alive = [True] * G
    terminal = longest = 0
    for move in range(case.moves):
        for i in range(case.count):
            if case.noise == "philox":
                buf = torch.full((G, batch, A), float("nan"), dtype=torch.float64, device="cuda")
                eng.select(batch, i, None, noise_out=buf)
                noise = buf.cpu().numpy()
                assert np.isfinite(noise).all() and (noise >= 0).all(), "device noise left unwritten or negative"
            else:
                noise = host_noise(case, rng)
                eng.select(batch, i, torch.from_numpy(noise).cuda())
            kind = eng.region("desc_kind")[:, :batch].cpu().numpy()
            plen = eng.region("desc_path_len")[:, :batch].cpu().numpy()
            live = np.array(alive)
            terminal += int((kind[live] == KIND_TERMINAL).sum())
            longest = max(longest, int(plen[live].max()) if live.any() else 0)
            eng.plan(batch)
            n = eng.leaf_count()
            planes = eng.leaf_planes(n).cpu().numpy()
            pri, val = stub(planes, A) if n else (np.zeros((1, A), np.float32), np.zeros(1, np.float32))
            eng.expand_backup(batch, torch.from_numpy(np.ascontiguousarray(pri)).cuda(),
                              torch.from_numpy(np.ascontiguousarray(val)).cuda())
            for g in range(G):
                if alive[g]:
                    trees[g][players[g] if tpg == 2 else 0].minibatch(batch, states[g], players[g], noise[g])
        for g in range(G):
            if not alive[g]:
                continue
            for t in range(tpg):
                errs = diff_tree(eng.export_tree(g * tpg + t), trees[g][t], A)
                assert not errs, "%s: game %d move %d tree %d: %s" % (case.name, g, move, t, errs[:5])
        pi_d, q_d, _ = eng.root_policy(2, case.tau_plies)
        pi_d, q_d = pi_d.cpu().numpy(), q_d.cpu().numpy()
        plies_dev = eng.region("ply").cpu().numpy()
        u = rng.random(G)
        actions = eng.advance(case.tau_plies, torch.from_numpy(u).cuda()).cpu().numpy()
        for g in range(G):
            if not alive[g]:
                assert actions[g] == -1
                continue
            tree = trees[g][players[g] if tpg == 2 else 0]
            pi, q = tree.get_policy_value(states[g], tau=1 if plies_dev[g] < case.tau_plies else 0)
            assert [float(x) for x in pi] == pi_d[g].tolist(), "%s: policy differs, game %d move %d" % (case.name, g, move)
            np.testing.assert_allclose(np.array([float(x) for x in q]), q_d[g], atol=1e-6)
            a = np_choice(pi, u[g])
            assert a == actions[g], "%s: sampled action differs, game %d move %d" % (case.name, g, move)
            states[g], won = og.move(states[g], a, players[g])
            players[g] = 1 - players[g]
            if won or not og.possible_moves(states[g]):
                alive[g] = False
        st_dev, pl_dev = eng.roots()
        status = eng.region("status").cpu().numpy()
        for g in range(G):
            assert st_dev[g] == states[g]
            assert (status[g] == 0) == alive[g]
            if alive[g]:
                assert pl_dev[g] == players[g]
    assert eng.counters()["errors"] == 0
    eng.close()
    return terminal, longest


@pytest.mark.parametrize("case", PARITY_CASES, ids=[c.name for c in PARITY_CASES])
def test_search_parity_matrix(torch_cuda, case):
    terminal, _ = run_case(torch_cuda, case)
    if case.A <= 16 or case.connect4:  # nearly full roots: wins and draws inside the search
        assert terminal > 0, "%s: no terminal descent" % case.name


@pytest.mark.parametrize("case", CHAIN_CASES, ids=[c.name for c in CHAIN_CASES])
def test_search_parity_deep_paths(torch_cuda, case):
    """Back-up paths longer than the 32 lanes of expand_backup_body's depth loop (two or three passes), with every
    descent of a 32-wide minibatch walking the same chain of edges."""
    _, longest = run_case(torch_cuda, case)
    assert longest > case.min_path, (case.name, longest)


@pytest.mark.parametrize("case", VL_CASES, ids=[c.name for c in VL_CASES])
def test_virtual_loss_matches_its_oracle(torch_cuda, case):
    run_case(torch_cuda, case)


@pytest.mark.parametrize("n", NOISE_BOARDS)
def test_device_noise_every_width(torch_cuda, n):
    """noise_kernel at every (GW, APL): the vectors are Dirichlet draws that sum to one, they are the addressed host
    stream of rng.cuh for every action (those at and beyond 32, 64 and 128 included), and at A = 36 and 225 their
    marginal mean and variance over 2 x 10^4 vectors are Dirichlet(0.3 x A)'s."""
    torch = torch_cuda
    from caro_ai_b200.engine import SelfPlayEngine
    from caro_ai_b200.game import TicTacToe
    from conftest import ROOT
    A = n * n
    moments = A in (36, 225)
    G, Bt, mb, seed = (2500 if moments else 256), 8, 3, 0x0123456789ABCDEF + n
    eng = SelfPlayEngine(TicTacToe(n, min(n, 5)), G, max_batch=Bt, node_capacity=16, seed=seed)
    out = torch.full((G, Bt, A), float("nan"), dtype=torch.float64, device="cuda")
    eng.select(Bt, mb, None, noise_out=out)
    z = out.cpu().numpy()
    assert np.isfinite(z).all() and (z >= 0).all()
    np.testing.assert_allclose(z.sum(axis=2), 1.0, atol=1e-12)
    so = os.path.join(ROOT, "tests", "native", "libhostcheck.so")
    if not os.path.exists(so):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC",
                               os.path.join(ROOT, "tests", "native", "hostcheck.cpp"), "-o", so])
    hc = C.CDLL(so)
    hc.hc_gamma.restype = C.c_float
    hc.hc_gamma.argtypes = [C.c_float] + [C.c_uint32] * 5
    uid = eng.region("uid").cpu().numpy().astype(np.uint64)
    ply = eng.region("ply").cpu().numpy()
    who = eng.region("root_player").cpu().numpy()
    k0, k1 = (seed & 0xFFFFFFFF) ^ 0x44495243, seed >> 32  # kStreamDirichlet (rng.cuh)
    close = np.zeros(A, np.int64)
    total = 0
    for g in range(0, G, max(1, G // 24)):
        c0 = int(uid[g]) & 0xFFFFFFFF
        c1 = ((int(uid[g]) >> 32) ^ (int(ply[g]) << 16) ^ int(who[g])) & 0xFFFFFFFF
        for j in range(Bt):
            gm = np.array([hc.hc_gamma(0.3, k0, k1, c0, c1, ((mb * Bt + j) << 8) | a) for a in range(A)], dtype=np.float32)
            want = gm.astype(np.float64) / gm.astype(np.float64).sum()
            close += np.abs(z[g, j] - want) <= 1e-4 * np.maximum(want, 1e-6) + 1e-9
            total += 1
    assert close.sum() >= 0.995 * total * A, (close.sum(), total * A)
    for edge in (32, 64, 128):  # the components that only the wider instances write
        if A > edge:
            assert close[edge:].sum() >= 0.995 * total * (A - edge), (edge, close[edge:].sum(), total * (A - edge))
    if moments:
        flat = z.reshape(-1, A)
        mean_var = (1 / A) * (1 - 1 / A) / (0.3 * A + 1)
        se = np.sqrt(mean_var / len(flat))
        assert np.abs(flat.mean(axis=0) - 1 / A).max() < 6 * se, (np.abs(flat.mean(axis=0) - 1 / A).max(), se)
        np.testing.assert_allclose(flat.var(axis=0).mean(), mean_var, rtol=0.03)
        for lo, hi in ((0, 32), (32, 64), (64, 128), (128, A)):  # every lane block of the group carries the variance
            hi = min(hi, A)
            if lo < hi:
                np.testing.assert_allclose(flat[:, lo:hi].var(axis=0).mean(), mean_var, rtol=0.1)
    eng.close()
