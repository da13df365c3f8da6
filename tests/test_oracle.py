"""The CPU oracle (oracle/lbc_oracle.py) against the golden vectors dumped from the unmodified reference."""
import numpy as np
import pytest
import torch

import lbc_oracle as orc
from lbc_testing import gold, rel_err


def _ref_models():
    """Plain torch construction in the reference's order, via the package's parameter containers
    (the package never computes with them) -- checks init parity too."""
    from learningbycheating_b200.common import _TrunkParams  # noqa: F401
    import learningbycheating_b200 as lbc
    torch.manual_seed(0)
    s = lbc.ImagePolicyModelSS('resnet34', all_branch=True)
    t = lbc.BirdViewPolicyModelSS('resnet18', all_branch=True)
    return s, t


def test_init_matches_reference():
    from lbc_testing import check_init
    s, t = _ref_models()
    check_init(s, "student")
    check_init(t, "teacher")
    init = gold("init_seed0.npz")
    assert [k for k, _ in s.named_parameters()] == list(init["student/param_names"])
    assert [k for k, _ in t.named_parameters()] == list(init["teacher/param_names"])


@pytest.fixture
def golden_threads():
    """The golden runs' intra-op thread count.  With another count the mathematically zero head gradients (softmax shift
    invariance) come out as different rounding noise, Adam's first step turns that noise into +-lr moves, and the later
    steps no longer replay."""
    from make_golden import GOLDEN_THREADS
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(n)


@pytest.mark.parametrize("phase", [0, 1])
def test_oracle_train_step_matches_golden(phase, golden_threads):
    s, t = _ref_models()
    g = gold("student_B2_phase%d.npz" % phase)
    b = orc.synthetic_batch(2)
    sd = orc.leafify(s.state_dict())
    td = {k: v.clone() for k, v in t.state_dict().items()}
    st = orc.new_adam_state()
    for step in range(2):
        o = orc.train_step(sd, td, b["rgb"], b["birdview"], b["speed"], b["command"], phase, adam_state=st)
        assert rel_err(o["pred"], g["step%d/pred" % step]) < 1e-5
        assert rel_err(o["preds"], g["step%d/preds" % step]) < 1e-5
        assert rel_err(o["loss"], g["step%d/loss" % step]) < 1e-5
        for k, gr in o["grads"].items():
            key = "step%d/grad/%s/full" % (step, k)
            if gr is not None and key in g.files and float(g["step%d/grad/%s/l2" % (step, k)]) > 1e-6:
                assert rel_err(gr, g[key]) < 2e-4, k
        for k in sd:
            key = "step%d/post/%s/full" % (step, k)
            if key in g.files:
                np.testing.assert_allclose(sd[k].detach().numpy(), g[key], rtol=0, atol=3e-6)


def test_oracle_birdview_step_matches_golden(golden_threads):
    _, t = _ref_models()
    g = gold("birdview_B2.npz")
    b = orc.synthetic_batch(2)
    sd = orc.leafify(t.state_dict())
    o = orc.birdview_train_step(sd, b["birdview"], b["location"], b["speed"], b["command"], adam_state=orc.new_adam_state())
    assert rel_err(o["pred"], g["step0/pred"]) < 1e-5
    assert abs(float(o["loss_mean"]) - float(g["step0/loss_mean"])) < 1e-6


def test_spatial_softmax_known_answers():
    """The known-answer check the reference left commented out (bird_view/models/common.py:192-201)."""
    ka = gold("spatial_softmax_known.npz")
    px, py = orc.spatial_grid(48, 48)
    for key in ka.files:
        i, j = map(int, key.split("_"))
        f = torch.zeros(48 * 48)
        f[i * 48 + j] = 100
        w = torch.softmax(f, 0)
        xy = torch.stack([(px * w).sum(), (py * w).sum()])
        np.testing.assert_allclose(xy.numpy(), ka[key].reshape(-1), atol=1e-6)


def test_one_hot_clamps():
    y = orc.one_hot(torch.tensor([1., 4., 0., 9.]))
    assert y.tolist() == [[1, 0, 0, 0], [0, 0, 0, 1], [1, 0, 0, 0], [0, 0, 0, 1]]
    import learningbycheating_b200 as lbc
    assert torch.equal(lbc.one_hot(torch.tensor([1., 4., 0., 9.])), y)


def test_reference_forward_agrees():
    """One train-mode forward of the unmodified reference's seed-0 student (oracle/make_golden.py reference_forward):
    the golden training run starts from it, and the oracle reproduces it from the same state, which the package's
    seed-0 construction matches bit for bit."""
    from make_golden import state_sha256
    ref = gold("reference_forward_B2.npz")
    s, _ = _ref_models()
    sd = s.state_dict()
    assert list(sd.keys()) == list(ref["state_keys"])
    for k, h in zip(ref["state_keys"], ref["state_sha256"]):
        assert state_sha256(sd[k]) == h, k
    g = gold("student_B2_phase0.npz")
    assert rel_err(ref["pred"], g["step0/pred"]) < 1e-5
    b = orc.synthetic_batch(2)
    o, os_, _ = orc.policy_forward(orc.leafify(sd), b["rgb"], b["speed"], orc.one_hot(b["command"]),
                                   "resnet34", True, True)
    assert rel_err(o.detach(), ref["pred"]) < 1e-5
    assert rel_err(os_.detach(), ref["preds"]) < 1e-5
