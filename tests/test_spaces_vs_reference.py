"""CPU: the drop-in classes expose the SAME gym spaces as the reference's classes for every constructor variant RLlib's
policy builder reads them from (`observation_space`, `action_space`, the joint / global / concatenated / continuous
variants; cleanup_new.py:90-169, harvest_new.py:85-130, cleanup_features.py:60-75, self_driving_car_accelerate.py:36-45,
two_stage_train.py:48-60,503-523).  No device is touched: the drop-in objects create their device batch lazily.

With a checkout of the original project (SSD_REFERENCE_ROOT) the reference's classes are built live; without one, their
spaces come from tests/golden/reference_spaces.json.  That file was recorded from the drop-in classes at a commit where
this live comparison had passed with their space code unchanged since (last changed in be37088, compared in befbbfb),
i.e. it holds the reference's spaces; no reference checkout was at hand when it was stored.  Re-record it with a checkout
present: `SSD_REFERENCE_ROOT=<checkout> SSD_RECORD_REFERENCE_SPACES=1 python -m pytest tests/test_spaces_vs_reference.py`.
"""
import json
import os

import numpy as np
import pytest

from oracle import ref_stubs

LIVE = ref_stubs.live_reference() is not None
RECORD = os.environ.get("SSD_RECORD_REFERENCE_SPACES") == "1"
STORED_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_spaces.json")


def plain(x):
    """desc() as it reads back from JSON (tuples -> lists)"""
    return json.loads(json.dumps(x))


@pytest.fixture
def reference(request):
    """The reference's side of the comparison for this test case: `get(key, live_fn)` returns the live value (recorded
    under `key` with SSD_RECORD_REFERENCE_SPACES=1) or the stored one."""
    stored = json.load(open(STORED_PATH)) if os.path.exists(STORED_PATH) else {}
    seen = {}

    def get(key, live_fn):
        key = "%s/%s" % (request.node.name, key)
        if LIVE:
            seen[key] = plain(live_fn())
            return seen[key]
        assert key in stored, "no stored reference value for %s" % key
        return stored[key]
    yield get
    if RECORD and LIVE:
        stored.update(seen)
        with open(STORED_PATH, "w") as f:
            f.write("{\n%s\n}\n" % ",\n".join("%s: %s" % (json.dumps(k), json.dumps(v)) for k, v in sorted(stored.items())))

ATTRS = ("observation_space", "action_space", "global_action_space", "global_observation_space",
         "concatenated_observation_space", "continuous_action_space")


def bounds(x):
    """Box bounds as float64 values: ["all", v] when every entry is v (exact), else the full list"""
    a = np.asarray(x, dtype=np.float64).ravel()
    if a.size and bool((a == a[0]).all()):
        return ["all", float(a[0])]
    return a.tolist()


def desc(sp):
    t = type(sp).__name__
    if t == "Dict":
        return ("Dict", {k: desc(sp[k]) for k in sorted(sp.keys())})
    if t == "Box":
        return ("Box", tuple(sp.shape), bounds(sp.low), bounds(sp.high), str(np.dtype(sp.dtype)))
    if t == "Discrete":
        return ("Discrete", int(sp.n))
    if t == "MultiDiscrete":
        return ("MultiDiscrete", np.asarray(sp.nvec).tolist())
    raise AssertionError("unexpected space type %s" % t)


def creators():
    from contracts_b200.utils.env_creator_functions import env_creator as my_creator, get_base_env_tag as my_tag
    import contracts_b200.contract.contract_list as my_cl
    if not LIVE:
        return None, None, None, my_creator, my_cl, my_tag
    ref_stubs.install(ref_stubs.live_reference())
    from utils.env_creator_functions import env_creator as ref_creator, get_base_env_tag as ref_tag
    import contract.contract_list as ref_cl
    return ref_creator, ref_cl, ref_tag, my_creator, my_cl, my_tag


BASES = [("CleanupNew", dict(num_agents=3, env_params={}, image_obs=True)),
         ("CleanupNew", dict(num_agents=8, env_params={}, image_obs=True, one_hot_id=True, disable_firing=False)),
         ("CleanupNew", dict(num_agents=2, env_params={}, image_obs=False)),
         ("HarvestNew", dict(num_agents=4, env_params={}, image_obs=True)),
         ("HarvestNew", dict(num_agents=5, env_params={}, image_obs=True, one_hot_id=True)),
         ("HarvestNew", dict(num_agents=4, env_params={}, image_obs=False, disable_firing=False)),
         ("Cleanup", dict(num_agents=5)), ("Harvest", dict(num_agents=3)), ("SelfDrive", dict(num_agents=4)),
         ("SelfDrive", dict(num_agents=2, low_bound=-5.0, high_bound=7.5))]
CONTRACT_OF = {"CleanupNew": "CleanupContract", "HarvestNew": "HarvestFeaturemodLocalContract", "Cleanup": "CleanupContract",
               "Harvest": "HarvestFeaturemodLocalContract", "SelfDrive": "SelfdriveContractDistprop"}


@pytest.mark.parametrize("tag,cfg", BASES, ids=["%s-%d" % (t, i) for i, (t, c) in enumerate(BASES)])
def test_base_env_spaces_match_reference(reference, tag, cfg):
    ref_creator, _, _, my_creator, _, _ = creators()
    r = [None]

    def ref_env():
        r[0] = r[0] or ref_creator(tag, dict(cfg))
        return r[0]
    m = my_creator(tag, dict(cfg))
    want = reference("spaces", lambda: {attr: desc(getattr(ref_env(), attr)) for attr in ATTRS if hasattr(ref_env(), attr)})
    seen = 0
    for attr in ATTRS:
        if attr in want:
            assert hasattr(m, attr), "%s: drop-in class lacks %s" % (tag, attr)
            assert plain(desc(getattr(m, attr))) == want[attr], "%s %r: %s differs" % (tag, cfg, attr)
            seen += 1
    assert seen >= 2
    assert m.num_agents == reference("num_agents", lambda: ref_env().num_agents)


@pytest.mark.parametrize("tag,cfg", BASES, ids=["%s-%d" % (t, i) for i, (t, c) in enumerate(BASES)])
def test_contract_wrapper_spaces_match_reference(reference, tag, cfg):
    """SeparateContractEnv.__init__ (two_stage_train.py:48-60): the observation gains the `contract` Box (image envs) or two
    more entries (flat observations); the contract's own space comes from contract_list.py."""
    ref_creator, ref_cl, _, my_creator, my_cl, _ = creators()
    n = cfg["num_agents"]
    conv = bool(cfg.get("image_obs"))

    def spaces(creator, cl):
        base = creator(tag, dict(cfg))
        contract = getattr(cl, CONTRACT_OF[tag])(n)
        env = creator("ContractWrapperSubgame", dict(num_agents=n, base_env=base, contract=contract, convolutional=conv))
        return plain((desc(env.observation_space), desc(env.action_space), desc(contract.contract_space)))
    assert spaces(my_creator, my_cl) == reference("spaces", lambda: spaces(ref_creator, ref_cl)), "%s %r" % (tag, cfg)


@pytest.mark.parametrize("kwargs", [dict(global_obs=True), dict(concatenated_obs=True)], ids=["global", "concatenated"])
@pytest.mark.parametrize("tag,n", [("CleanupNew", 2), ("HarvestNew", 4)])
def test_joint_env_spaces_match_reference(reference, tag, n, kwargs):
    ref_creator, _, _, my_creator, _, _ = creators()

    def spaces(creator):
        base = creator(tag, dict(num_agents=n, env_params={}, image_obs=True))
        env = creator("JointEnv", dict(base_env=base, num_agents=n, **kwargs))
        return plain((desc(env.observation_space), desc(env.action_space)))
    assert spaces(my_creator) == reference("spaces", lambda: spaces(ref_creator))


def test_base_env_tags_match_reference(reference):
    _, _, ref_tag, _, _, my_tag = creators()
    for name in ("selfdrive", "harvest", "harvest_new", "cleanup", "cleanup_new"):
        assert my_tag({"environment": name}) == reference(name, lambda: ref_tag({"environment": name}))
    if LIVE:
        with pytest.raises(AssertionError):
            ref_tag({"environment": "nope"})
    with pytest.raises(AssertionError):
        my_tag({"environment": "nope"})
