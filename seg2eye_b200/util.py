"""Checkpoint helpers with the reference's on-disk layout (util/util.py:195-221):
`<checkpoints_dir>/<name>/<epoch>_net_<G|D|E>.pth` = fp32 CPU state_dict with the reference's keys."""
import os

import torch

from . import ops


def save_network(net, label, epoch, opt):
    save_path = os.path.join(opt.checkpoints_dir, opt.name, '%s_net_%s.pth' % (epoch, label))
    os.makedirs(os.path.dirname(save_path), exist_ok=True)
    sd = {k: v.detach().to('cpu') for k, v in net.state_dict().items()}
    torch.save(sd, save_path)


def load_network(net, label, epoch, opt, save_dir=None):
    if save_dir is None:
        save_dir = os.path.join(opt.checkpoints_dir, opt.name)
    save_path = os.path.join(save_dir, '%s_net_%s.pth' % (epoch, label))
    weights = torch.load(save_path, map_location='cpu')
    # checkpoints written by the reference under nn.DataParallel carry a 'module.' prefix
    weights = {(k[len('module.'):] if k.startswith('module.') else k): v for k, v in weights.items()}
    net.load_state_dict(weights)
    ops.bump_weights_epoch()
    print(f"Loaded network from {save_path} for epoch {epoch}")
    return net


def _named_params(nets):
    """'G.fc.weight' style names for the parameters of the (tag, network) pairs, in optimizer order."""
    return [("%s.%s" % (tag, n), p_) for tag, net in nets if net is not None for n, p_ in net.named_parameters()]


def save_optimizer(optimizer, label, epoch, opt, nets, extra=None):
    """Beyond the reference (which restarts Adam from zero moments on --continue_train, util/util.py:195-221 saves
    networks only): `<epoch>_optim_<G|D>.pth` next to the network files -- fp32 CPU tensors keyed by parameter NAME
    ('G.up_0.conv_0.weight_orig': {'exp_avg', 'exp_avg_sq'}), plus the step count and learning rate.  Files the reference
    never reads; its own checkpoints are untouched.  `extra`: further top-level entries of the file (the trainer stores the
    --diff_augment generator state under 'diffaug' in the D file)."""
    save_path = os.path.join(opt.checkpoints_dir, opt.name, '%s_optim_%s.pth' % (epoch, label))
    os.makedirs(os.path.dirname(save_path), exist_ok=True)
    names = {id(p_): n for n, p_ in _named_params(nets)}
    out = {"state": {}, "groups": []}
    for group in optimizer.param_groups:
        st = group.get('_s2e_state')
        out["groups"].append({"lr": group['lr'], "betas": tuple(group['betas']), "eps": group['eps'],
                              "weight_decay": group['weight_decay'], "step": float(st[0]) if st is not None else 0.0})
        for p_ in group['params']:
            s_ = optimizer.state.get(p_)
            if s_:
                out["state"][names[id(p_)]] = {k: s_[k].detach().to('cpu') for k in ('exp_avg', 'exp_avg_sq')}
    out.update(extra or {})
    torch.save(out, save_path)


def load_optimizer_entry(label, epoch, opt, key):
    """Top-level entry `key` of the file save_optimizer wrote (None when the file or the entry does not exist)."""
    path = os.path.join(opt.checkpoints_dir, opt.name, '%s_optim_%s.pth' % (epoch, label))
    if not os.path.exists(path):
        return None
    return torch.load(path, map_location='cpu').get(key)


def load_optimizer(optimizer, label, epoch, opt, nets):
    """Restore what save_optimizer wrote; returns False (and leaves the optimizer fresh, like the reference) if the file
    does not exist."""
    path = os.path.join(opt.checkpoints_dir, opt.name, '%s_optim_%s.pth' % (epoch, label))
    if not os.path.exists(path):
        return False
    blob = torch.load(path, map_location='cpu')
    params = dict(_named_params(nets))
    for name, s_ in blob["state"].items():
        p_ = params[name]
        optimizer.state[p_] = {k: v.to(device=p_.device, dtype=torch.float32).clone() for k, v in s_.items()}
    for group, g in zip(optimizer.param_groups, blob["groups"]):
        group['lr'] = g["lr"]
        dev = group['params'][0].device
        group['_s2e_state'] = torch.tensor([g["step"], g["lr"], 0.0, 0.0], dtype=torch.float32, device=dev)
        group['_s2e_lr'] = g["lr"]
    print(f"Loaded optimizer state from {path}")
    return True
