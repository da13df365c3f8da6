"""TEST INFRASTRUCTURE ONLY -- generate tests/golden/*.npz from the UNMODIFIED reference.

Needs the reference tree (LBC_REFERENCE_ROOT, see ref_import.py):   python oracle/make_golden.py [reference_forward]
(with the argument, only tests/golden/reference_forward_B2.npz is rewritten).

For each case it drives the reference's own classes (ImagePolicyModelSS, BirdViewPolicyModelSS,
train_image_phase{0,1}.CoordConverter / LocationLoss, torch.optim.Adam) exactly as
train_or_eval does (training/train_image_phase0.py:166-185, train_image_phase1.py:174-205,
train_birdview.py:116-129), records outputs, and asserts that oracle/lbc_oracle.py (the
restatement that travels to the GPU box) reproduces them.  Protocol = SURVEY.md 8(c).
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import lbc_oracle as orc  # noqa: E402
import ref_import  # noqa: E402

OUT = os.path.join(HERE, "..", "tests", "golden")
N_STEPS = 3
SMALL = 4096
# torch's CPU kernels split their reductions by intra-op thread, so the last bits of a result depend on the thread count;
# the golden runs were recorded with this many, and tests that replay them bit for bit set it too
GOLDEN_THREADS = 8


def sample_coords(shape, k=24, seed=7):
    rng = np.random.RandomState(seed)
    return np.stack([rng.randint(0, s, size=k) for s in shape], 1)


def tap_summary(t):
    a = t.double().numpy()
    coords = sample_coords(a.shape)
    vals = a[tuple(coords.T)]
    return dict(mean=a.mean(), absmean=np.abs(a).mean(), sqmean=(a * a).mean(),
                coords=coords, vals=vals, shape=np.array(a.shape))


def tensor_summary(prefix, name, t, out):
    a = t.detach().double().numpy().reshape(-1)
    out["%s/%s/l2" % (prefix, name)] = np.sqrt((a * a).sum())
    out["%s/%s/sum" % (prefix, name)] = a.sum()
    out["%s/%s/head" % (prefix, name)] = a[:8].copy()
    if a.size <= SMALL:
        out["%s/%s/full" % (prefix, name)] = t.detach().float().numpy().copy()


def run_case(ns, B, phase, student0, teacher0):
    """phase 0/1: student training against the frozen teacher."""
    torch.manual_seed(1234)
    batch = orc.synthetic_batch(B, seed=1)
    student = ns.ImagePolicyModelSS('resnet34', all_branch=True)
    student.load_state_dict(student0)
    teacher = ns.BirdViewPolicyModelSS('resnet18', all_branch=True)
    teacher.load_state_dict(teacher0)
    student.train()
    teacher.eval()
    optim = torch.optim.Adam(student.parameters(), lr=1e-4)
    if phase == 0:
        conv = ns.phase0.CoordConverter(w=384, h=160, fov=90, world_y=1.4, fixed_offset=4.0, device='cpu')
        crit = ns.phase0.LocationLoss(w=384, h=160, device='cpu')
    else:
        conv = ns.phase1.CoordConverter(w=384, h=160, fov=90, world_y=1.4, fixed_offset=4.0, device='cpu')
        crit = ns.phase1.LocationLoss()

    # restatement state
    o_student = orc.leafify(student0)
    o_teacher = {k: v.clone() for k, v in teacher0.items()}
    o_adam = orc.new_adam_state()

    out = {}
    names = [k for k, _ in student.named_parameters()]
    for step in range(N_STEPS):
        oh = ns.one_hot(batch["command"])
        with torch.no_grad():
            t_pred, t_preds = teacher(batch["birdview"], batch["speed"], oh)
        pred, preds = student(batch["rgb"], batch["speed"], oh)
        if phase == 0:
            target = conv(t_pred)
            loss = crit(pred, target)
        else:
            target = None
            loss = crit(conv(preds), t_preds)
        loss_mean = loss.mean()
        optim.zero_grad()
        loss_mean.backward()
        grads = {k: (p.grad.clone() if p.grad is not None else None) for k, p in student.named_parameters()}
        optim.step()

        taps = {} if step == 0 else None
        o = orc.train_step(o_student, o_teacher, batch["rgb"], batch["birdview"], batch["speed"],
                           batch["command"], phase, adam_state=o_adam, taps=taps)
        # ---- restatement == reference ----
        def chk(a, b, what, tol=2e-6):
            d = (a.double() - b.double()).abs().max().item()
            s = b.double().abs().max().item() + 1e-30
            assert d <= tol * max(1.0, s), "restatement mismatch %s: %g (scale %g)" % (what, d, s)
        chk(o["pred"], pred, "pred")
        chk(o["preds"], preds, "preds")
        chk(o["t_pred"], t_pred, "t_pred")
        chk(o["loss"], loss, "loss", 1e-5)
        for k in names:
            if grads[k] is None:
                assert o["grads"][k] is None
            else:
                chk(o["grads"][k], grads[k], "grad " + k, 2e-5)
        sd_now = student.state_dict()
        for k in sd_now:
            if sd_now[k].dtype.is_floating_point:
                chk(o_student[k].detach(), sd_now[k], "post-step " + k, 2e-6)
            else:
                assert int(o_student[k]) == int(sd_now[k]), k

        s = "step%d" % step
        out[s + "/pred"] = pred.detach().numpy().copy()
        out[s + "/preds"] = preds.detach().numpy().copy()
        out[s + "/t_pred"] = t_pred.numpy().copy()
        out[s + "/t_preds"] = t_preds.numpy().copy()
        out[s + "/loss"] = loss.detach().numpy().copy()
        out[s + "/loss_mean"] = np.float64(loss_mean.item())
        if target is not None:
            out[s + "/target_px"] = target.numpy().copy()
        gl2 = 0.0
        for k in names:
            if grads[k] is None:
                continue
            tensor_summary(s + "/grad", k, grads[k], out)
            gl2 += float((grads[k].double() ** 2).sum())
        out[s + "/grad_global_l2"] = np.float64(np.sqrt(gl2))
        for k, v in sd_now.items():
            if v.dtype.is_floating_point and not k.endswith(("pos_x", "pos_y")):
                tensor_summary(s + "/post", k, v, out)
            elif not v.dtype.is_floating_point:
                out[s + "/post/" + k] = np.int64(int(v))
        if taps is not None:
            for k, t in taps.items():
                for kk, vv in tap_summary(t).items():
                    out["step0/tap/%s/%s" % (k, kk)] = vv
        print("  B=%d phase=%d step=%d loss=%.8f" % (B, phase, step, loss_mean.item()), flush=True)
    out["B"] = np.int64(B)
    out["phase"] = np.int64(phase)
    return out


def run_birdview_case(ns, B, teacher0):
    """config 5: train_birdview.py step (teacher architecture in train mode, L1 vs dataset locations)."""
    batch = orc.synthetic_batch(B, seed=1)
    net = ns.BirdViewPolicyModelSS('resnet18')
    net.load_state_dict(teacher0)
    net.train()
    optim = torch.optim.Adam(net.parameters(), lr=1e-4)
    crit = ns.birdview.LocationLoss(w=192, h=192, choice='l1')
    o_sd = orc.leafify(teacher0)
    o_adam = orc.new_adam_state()
    out = {}
    names = [k for k, _ in net.named_parameters()]
    for step in range(N_STEPS):
        oh = ns.one_hot(batch["command"])
        pred = net(batch["birdview"], batch["speed"], oh)
        loss = crit(pred, batch["location"])
        loss_mean = loss.mean()
        optim.zero_grad()
        loss_mean.backward()
        grads = {k: (p.grad.clone() if p.grad is not None else None) for k, p in net.named_parameters()}
        optim.step()
        o = orc.birdview_train_step(o_sd, batch["birdview"], batch["location"], batch["speed"],
                                    batch["command"], adam_state=o_adam)
        assert (o["pred"] - pred.detach()).abs().max() < 2e-6
        assert (o["loss"] - loss.detach()).abs().max() < 1e-5
        sd_now = net.state_dict()
        for k in sd_now:
            if sd_now[k].dtype.is_floating_point:
                assert (o_sd[k].detach() - sd_now[k]).abs().max() < 2e-6, k
        s = "step%d" % step
        out[s + "/pred"] = pred.detach().numpy().copy()
        out[s + "/loss"] = loss.detach().numpy().copy()
        out[s + "/loss_mean"] = np.float64(loss_mean.item())
        gl2 = 0.0
        for k in names:
            if grads[k] is None:
                continue
            tensor_summary(s + "/grad", k, grads[k], out)
            gl2 += float((grads[k].double() ** 2).sum())
        out[s + "/grad_global_l2"] = np.float64(np.sqrt(gl2))
        for k, v in sd_now.items():
            if v.dtype.is_floating_point and not k.endswith(("pos_x", "pos_y")):
                tensor_summary(s + "/post", k, v, out)
        print("  birdview B=%d step=%d loss=%.8f" % (B, step, loss_mean.item()), flush=True)
    out["B"] = np.int64(B)
    return out


def state_sha256(t):
    """Digest of a state_dict tensor's bytes: tests hold the package's initial state to the reference's, bit for bit."""
    import hashlib
    return hashlib.sha256(t.detach().contiguous().cpu().numpy().tobytes()).hexdigest()


def reference_forward(ns):
    """One train-mode forward of the reference's seed-0 student on synthetic_batch(2): its predictions, and a digest of
    every state_dict tensor it was computed from."""
    torch.manual_seed(0)
    s = ns.ImagePolicyModelSS('resnet34', all_branch=True)
    sd = s.state_dict()
    keys, digests = np.array(list(sd.keys())), np.array([state_sha256(v) for v in sd.values()])   # before the forward
    b = orc.synthetic_batch(2)                                                                     # updates BN buffers
    s.train()
    pred, preds = s(b["rgb"], b["speed"], ns.one_hot(b["command"]))
    np.savez_compressed(os.path.join(OUT, "reference_forward_B2.npz"), pred=pred.detach().numpy().copy(),
                        preds=preds.detach().numpy().copy(), state_keys=keys, state_sha256=digests)
    print("reference forward written")


def main(only=None):
    ns = ref_import.load()
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(GOLDEN_THREADS)
    if only == "reference_forward":
        reference_forward(ns)
        return
    reference_forward(ns)
    torch.manual_seed(0)     # SURVEY 8(c): student first, then teacher (RNG order matters)
    student = ns.ImagePolicyModelSS('resnet34', all_branch=True)
    teacher = ns.BirdViewPolicyModelSS('resnet18', all_branch=True)
    student0 = {k: v.clone() for k, v in student.state_dict().items()}
    teacher0 = {k: v.clone() for k, v in teacher.state_dict().items()}

    init = {}
    for tag, sd in (("student", student0), ("teacher", teacher0)):
        init[tag + "/keys"] = np.array(list(sd.keys()))
        init[tag + "/shapes"] = np.array([str(tuple(v.shape)) for v in sd.values()])
        for k, v in sd.items():
            if v.dtype.is_floating_point:
                a = v.double().numpy().reshape(-1)
                init["%s/%s/sum" % (tag, k)] = a.sum()
                init["%s/%s/abssum" % (tag, k)] = np.abs(a).sum()
                init["%s/%s/head" % (tag, k)] = a[:8].copy()
    init["student/param_names"] = np.array([k for k, _ in student.named_parameters()])
    init["teacher/param_names"] = np.array([k for k, _ in teacher.named_parameters()])
    np.savez_compressed(os.path.join(OUT, "init_seed0.npz"), **init)
    print("init checksums written")

    # SpatialSoftmax known-answer snippet the reference left commented out (common.py:192-201)
    ss = ns.common.SpatialSoftmax(48, 48, 1)
    ka = {}
    for (i, j) in [(47, 0), (47, 24), (47, 47), (0, 24)]:
        f = np.zeros((48, 48), np.float32)
        f[i, j] = 100
        ka["%d_%d" % (i, j)] = ss(torch.from_numpy(f)[None, None]).numpy().copy()
    np.savez_compressed(os.path.join(OUT, "spatial_softmax_known.npz"), **ka)

    for B in (2, 4):
        for phase in (0, 1):
            print("case B=%d phase=%d" % (B, phase), flush=True)
            out = run_case(ns, B, phase, student0, teacher0)
            np.savez_compressed(os.path.join(OUT, "student_B%d_phase%d.npz" % (B, phase)), **out)
    out = run_birdview_case(ns, 2, teacher0)
    np.savez_compressed(os.path.join(OUT, "birdview_B2.npz"), **out)
    print("done")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else None)
