"""SelfAcceleratingCarEnv + SelfdriveContractDistprop (self_driving_car_accelerate.py:49-250,
contract_list.py:66-102): the reference's golden episodes (tests/golden/selfdrive_*.npz) replayed through the C
oracle on CPU and through the CUDA path on GPU.  Everything is float64 and compared bit-exactly (the north star's
fp32 tolerance is not needed: the <= 8-car kinematics run in fp64 on the device)."""
import numpy as np
import pytest

import golden_util as gu

NAMES = gu.fixture_names("selfdrive_")


def test_selfdrive_fixtures_present():
    assert len(NAMES) >= 5


class _OracleCar:
    def __init__(self, oracle_mod, fx):
        self.o = oracle_mod.CarOracle(1, int(fx["n"]), contract=bool(fx["contract"]), seed=int(fx["seed"]),
                                      first_env_id=int(fx["env_id"]))

    def reset(self):
        obs = self.o.reset()[0]
        return obs, self.o.get_state()["theta"][0]

    def step(self, a):
        r = self.o.step(np.asarray(a)[None])
        st = self.o.get_state()
        out = {k: v[0] for k, v in r.items()}
        out.update(pos=st["pos"][0], vel=st["vel"][0], metric_transfers=st["transfers"][0])
        return out


class _CudaCar:
    def __init__(self, fx, E=5, index=3):
        from contracts_b200.selfdrive import BatchedCarEnv
        self.i = index
        self.env = BatchedCarEnv(E, int(fx["n"]), contract="SelfdriveContractDistprop" if bool(fx["contract"]) else None,
                                 seed=int(fx["seed"]), first_env_id=(int(fx["env_id"]) - index) & 0xFFFFFFFF)

    def reset(self):
        obs = self.env.reset()[self.i].cpu().numpy()
        return obs, self.env.get_state()["theta"][self.i].item()

    def step(self, a):
        import torch
        acts = torch.zeros((self.env.E, self.env.n), dtype=torch.float32)
        acts[:] = torch.as_tensor(np.asarray(a, dtype=np.float32))
        obs, rew, done, info = self.env.step(acts.cuda())
        st = self.env.get_state()
        i = self.i
        return {"obs": obs[i].cpu().numpy(), "rew": rew[i].cpu().numpy(), "base_rew": self.env.base_rew[i].cpu().numpy(),
                "transfers": self.env.transfers[i].cpu().numpy(), "info": info[i].cpu().numpy(),
                "done": done[i].cpu().numpy(), "pos": st["pos"][i].cpu().numpy(), "vel": st["vel"][i].cpu().numpy(),
                "metric_transfers": st["transfers"][i].item()}


def replay(backend, fx):
    n = int(fx["n"])
    wrapped = bool(fx["contract"])
    D = 2 * (n + 1) + 3
    for ep in range(fx["actions"].shape[0]):
        obs, theta = backend.reset()
        ctx = "reset ep %d" % ep
        gu.assert_same("reset obs", obs, fx["reset_obs"][ep][:, :D], ctx)
        if wrapped:
            gu.assert_same("theta", theta, fx["reset_theta"][ep], ctx)
            gu.assert_same("obs theta", fx["reset_obs"][ep][:, D], np.full(n, theta), ctx)
        for t in range(int(fx["length"][ep])):
            ctx = "ep %d step %d" % (ep, t)
            o = backend.step(fx["actions"][ep, t])
            act = fx["active"][ep, t].astype(bool)
            gu.assert_same("active", o["info"][:, 1], fx["active"][ep, t], ctx)
            gu.assert_same("obs", o["obs"][act], fx["obs"][ep, t][act][:, :D], ctx)
            gu.assert_same("rew", o["rew"][act], fx["rew"][ep, t][act], ctx)
            gu.assert_same("done", o["done"], fx["done"][ep, t], ctx)
            gu.assert_same("just_passed", o["info"][:, 0], fx["just_passed"][ep, t], ctx)
            first = int(np.argmax(act))
            gu.assert_same("ambulance_rank", o["info"][first, 2], fx["ambulance_rank"][ep, t], ctx)
            gu.assert_same("ambulance_dist_to_front", o["info"][first, 3], fx["ambulance_dist_to_front"][ep, t], ctx)
            gu.assert_same("pos", o["pos"], fx["pos"][ep, t], ctx)
            gu.assert_same("vel", o["vel"], fx["vel"][ep, t], ctx)
            if wrapped:
                gu.assert_same("base_rew", o["base_rew"][act], fx["base_rew"][ep, t][act], ctx)
                gu.assert_same("transfers", o["transfers"], fx["transfers"][ep, t], ctx)
                gu.assert_same("metric transfers", o["metric_transfers"], fx["metric_transfers"][ep, t], ctx)


@pytest.mark.parametrize("name", NAMES)
def test_oracle_selfdrive_matches_reference(oracle_lib, name):
    replay(_OracleCar(oracle_lib, gu.load(name)), gu.load(name))


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_cuda_selfdrive_matches_reference(name):
    replay(_CudaCar(gu.load(name)), gu.load(name))


@pytest.mark.gpu
@pytest.mark.parametrize("name", [n for n in NAMES if "nocontract" not in n and n != "selfdrive_n1"])
def test_dropin_selfdrive_dict_api(name):
    """env_creator('SelfDrive') + ContractWrapperSubgame(SelfdriveContractDistprop), the reference's flat obs layout."""
    from contracts_b200.contract import contract_list
    from contracts_b200.utils.env_creator_functions import env_creator, get_base_env_tag
    fx = gu.load(name)
    n = int(fx["n"])
    base = env_creator(get_base_env_tag({"environment": "selfdrive"}), dict(num_agents=n, seed=int(fx["seed"]), env_id=int(fx["env_id"])))
    env = env_creator("ContractWrapperSubgame", dict(num_agents=n, base_env=base, contract=contract_list.SelfdriveContractDistprop(n),
                                                     convolutional=False))
    keys = ["a%d" % i for i in range(n)]
    assert env.observation_space.shape == (2 * (n + 1) + 3 + 2,)
    for ep in range(fx["actions"].shape[0]):
        obs = env.reset()
        gu.assert_same("reset obs", np.stack([obs[k] for k in keys]), fx["reset_obs"][ep], "ep %d" % ep)
        for t in range(int(fx["length"][ep])):
            ctx = "ep %d step %d" % (ep, t)
            acting = [k for i, k in enumerate(keys) if fx["active"][ep, t][i]]
            obs, rew, done, info = env.step({k: np.array([fx["actions"][ep, t][int(k[1:])]]) for k in acting})
            assert sorted(obs.keys()) == acting and sorted(rew.keys()) == acting, ctx
            for k in acting:
                i = int(k[1:])
                gu.assert_same("obs", obs[k], fx["obs"][ep, t][i], ctx)
                gu.assert_same("rew", rew[k], fx["rew"][ep, t][i], ctx)
                assert info[k]["just_passed"] == bool(fx["just_passed"][ep, t][i]), ctx
            gu.assert_same("done", [done[k] for k in keys] + [done["__all__"]], fx["done"][ep, t], ctx)
            gu.assert_same("ambulance_rank", info[acting[0]]["ambulance_rank"], fx["ambulance_rank"][ep, t], ctx)
            gu.assert_same("metric", base.metrics["transfers"], fx["metric_transfers"][ep, t], ctx)


@pytest.mark.gpu
@pytest.mark.parametrize("n,E,contract,params", [
    pytest.param(8, 4099, True, {}, id="8-4099-True"), pytest.param(3, 515, True, {}, id="3-515-True"),
    pytest.param(5, 130, False, {}, id="5-130-False"),
    # the non-default road and speed parameters that test_deep_differential.py pins reference -> oracle
    pytest.param(5, 777, True, dict(low_bound=-4.5, high_bound=6.25, start_vel=0.35, start_vel_ambulance=0.55), id="5-777-True-params"),
    pytest.param(3, 301, True, dict(low_bound=-20.0, high_bound=3.0, start_vel=0.05, start_vel_ambulance=1.0), id="3-301-True-params")])
def test_cuda_selfdrive_rollout_matches_oracle(oracle_lib, n, E, contract, params):
    """Random rollouts, every output, bit-exact, incl. masked re-resets of finished envs."""
    import torch
    from contracts_b200.selfdrive import BatchedCarEnv
    env = BatchedCarEnv(E, n, contract="SelfdriveContractDistprop" if contract else None, seed=7, first_env_id=123, **params)
    orc = oracle_lib.CarOracle(E, n, contract=contract, seed=7, first_env_id=123, **params)
    gu.assert_same("reset obs", env.reset().cpu().numpy(), orc.reset(), "reset")
    rng = np.random.RandomState(n)
    for t in range(260):
        a = (rng.uniform(-0.7, 1.0, size=(E, n)) * 0.15).astype(np.float32)
        o = orc.step(a)
        obs, rew, done, info = env.step(torch.from_numpy(a).cuda())
        ctx = "step %d" % t
        gu.assert_same("obs", obs.cpu().numpy(), o["obs"], ctx)
        gu.assert_same("rew", rew.cpu().numpy(), o["rew"], ctx)
        gu.assert_same("base_rew", env.base_rew.cpu().numpy(), o["base_rew"], ctx)
        gu.assert_same("transfers", env.transfers.cpu().numpy(), o["transfers"], ctx)
        gu.assert_same("info", info.cpu().numpy(), o["info"], ctx)
        gu.assert_same("done", done.cpu().numpy(), o["done"], ctx)
        fin = o["done"][:, -1].astype(bool)
        if t % 9 == 0 and fin.any():
            mask = fin.astype(np.uint8)
            r1 = env.reset(torch.from_numpy(mask).cuda()).cpu().numpy()
            r2 = orc.reset(mask)
            gu.assert_same("masked reset obs", r1[fin], r2[fin], ctx)
    so, sc = orc.get_state(), env.get_state()
    for k in ("pos", "vel", "theta", "transfers", "t"):
        gu.assert_same(k, sc[k].cpu().numpy(), so[k], "end")


@pytest.mark.gpu
def test_selfdrive_next_step_auto_reset():
    """ssd_selfdrive_io.auto_reset: an env whose episode ended is reset by the NEXT step call — compared env by env with
    single-env handles driven by explicit reset() (episodes end at different steps in different envs)."""
    import torch
    from contracts_b200.selfdrive import BatchedCarEnv
    E, n = 10, 4
    batch = BatchedCarEnv(E, n, contract="SelfdriveContractDistprop", seed=9, first_env_id=20)
    singles = [BatchedCarEnv(1, n, contract="SelfdriveContractDistprop", seed=9, first_env_id=20 + e) for e in range(E)]
    obs = batch.reset().cpu().numpy().copy()
    for e, s in enumerate(singles):
        assert np.array_equal(s.reset().cpu().numpy()[0], obs[e])
    rng = np.random.RandomState(2)
    done_prev = np.zeros(E, dtype=bool)
    resets = 0
    for t in range(500):
        acts = (rng.uniform(-0.02, 0.1, size=(E, n))).astype(np.float32)
        o, r, d, _ = batch.step(torch.as_tensor(acts).cuda(), auto_reset=True)
        o, r, d = o.cpu().numpy(), r.cpu().numpy(), d.cpu().numpy()
        for e, s in enumerate(singles):
            if done_prev[e]:
                so = s.reset().cpu().numpy()[0]
                resets += 1
                assert np.array_equal(o[e], so) and not r[e].any() and not d[e].any(), (t, e)
            else:
                so, sr, sd, _ = s.step(torch.as_tensor(acts[e:e + 1]).cuda())
                assert np.array_equal(o[e].view(np.uint64), so.cpu().numpy()[0].view(np.uint64)), (t, e)
                assert np.array_equal(r[e].view(np.uint64), sr.cpu().numpy()[0].view(np.uint64)), (t, e)
                assert np.array_equal(d[e], sd.cpu().numpy()[0])
        done_prev = d[:, n].astype(bool)
    assert resets >= E


@pytest.mark.gpu
@pytest.mark.parametrize("n,E,contract", [(8, 2050, True), (3, 333, True), (5, 64, False)])
def test_selfdrive_step_host_async_equals_step(n, E, contract):
    """ssd_selfdrive_step_host_async / ssd_step_host_wait: float32 host actions in, the compact result block out (int8
    rewards + exact float64 records + dones [E, n+1]) — bit for bit what ssd_selfdrive_step produces, auto-reset on."""
    import torch
    from contracts_b200.selfdrive import BatchedCarEnv
    c = "SelfdriveContractDistprop" if contract else None
    a = BatchedCarEnv(E, n, contract=c, seed=5, first_env_id=3)
    b = BatchedCarEnv(E, n, contract=c, seed=5, first_env_id=3)
    a.reset(); b.reset()
    rng = np.random.RandomState(4)
    T = 200
    acts = [torch.as_tensor((rng.uniform(-0.7, 1.0, size=(E, n)) * 0.15).astype(np.float32)).pin_memory() for _ in range(T)]
    res = [b.new_host_result(), b.new_host_result()]
    want = []
    for t in range(T):
        obs_a, rew_a, done_a, _ = a.step(acts[t].cuda(), auto_reset=True)
        want.append((rew_a.cpu().numpy().copy(), done_a.cpu().numpy().copy(), obs_a.cpu().numpy().copy() if t % 19 == 0 else None))
    tickets, sparse_total, finished = [], 0, 0

    def check(t):
        nonlocal sparse_total, finished
        b.step_host_wait(tickets[t])
        r = res[t & 1]
        assert np.array_equal(r.rewards().view(np.uint64), want[t][0].view(np.uint64)), t
        assert np.array_equal(r.done, want[t][1]), t
        w = want[t][0]
        fits = (w == np.round(w)) & (np.abs(w) <= 127) & ~(np.signbit(w) & (w == 0))
        assert np.array_equal(np.sort(r.rec_env[:r.count]), np.nonzero(~fits.all(1))[0]), t
        sparse_total += r.count
        finished += int(want[t][1][:, n].sum())
    for t in range(T):
        tickets.append(b.step_host_async(acts[t], res[t & 1], auto_reset=True))
        if want[t][2] is not None:
            assert np.array_equal(b.obs.cpu().numpy().view(np.uint64), want[t][2].view(np.uint64)), t
        if t >= 1:
            check(t - 1)
    check(T - 1)
    assert finished > 0
    assert (sparse_total > 0) == bool(contract)
