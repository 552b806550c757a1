"""SAC on the batched GPU env with nothing leaving the device: env step (fused CUDA kernel), VecNormalize statistics + replay
buffer with on-device sampling (`glgym.replay.DeviceReplayBuffer`, csrc/glg_replay.cuh), and a squashed-Gaussian actor, twin
critics, target networks and automatic entropy tuning in plain torch -- the off-policy counterpart of
examples/ppo_device_rollout.py, replacing `SubprocVecEnv -> VecMonitor -> VecNormalize -> SAC` (gl_gym/RL/utils.py:44-69).
The reference's configs/agents/sac.yml is not part of this tree, so the hyper-parameters are SB3 2.6.0's SAC defaults:
256x2 ReLU MLPs, lr 3e-4, buffer 1e6 transitions, batch 256, tau 0.005, gamma 0.99, learning_starts 100, train_freq 1 (one
vector step of all envs) and one gradient step per step, target entropy -6.  A demonstration of the data path, not a learning
claim: it prints env-steps/s including the updates.

    python examples/sac_device_replay.py [--n-envs 4096] [--iters 50] [--batch 256]
"""
import argparse, copy, os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "greenlight-gym2_b200"))
import torch
import torch.nn.functional as F
from glgym.replay import DeviceReplayBuffer
from glgym.vec_env import GreenLightVecEnv

ap = argparse.ArgumentParser()
ap.add_argument("--n-envs", type=int, default=4096)
ap.add_argument("--iters", type=int, default=50)
ap.add_argument("--batch", type=int, default=256)
ap.add_argument("--buffer-size", type=int, default=1_000_000)
ap.add_argument("--learning-starts", type=int, default=100)
ap.add_argument("--lr", type=float, default=3e-4)
ap.add_argument("--uncertainty-scale", type=float, default=0.0)
a = ap.parse_args()
dev = torch.device("cuda", 0)
torch.manual_seed(0)
GAMMA, TAU, NA = 0.99, 0.005, 6


def mlp(i, o):
    return torch.nn.Sequential(torch.nn.Linear(i, 256), torch.nn.ReLU(), torch.nn.Linear(256, 256), torch.nn.ReLU(), torch.nn.Linear(256, o))


class Actor(torch.nn.Module):
    def __init__(self, d):
        super().__init__()
        self.body = mlp(d, 2 * NA)

    def forward(self, obs):
        """Squashed Gaussian: action in (-1, 1) and its log-probability (SB3 SquashedDiagGaussianDistribution)."""
        mean, log_std = self.body(obs).chunk(2, dim=-1)
        std = log_std.clamp(-20, 2).exp()
        u = mean + std * torch.randn_like(mean)
        act = torch.tanh(u)
        logp = (-0.5 * ((u - mean) / std) ** 2 - std.log() - 0.9189385332046727).sum(-1)
        return act, logp - torch.log(1 - act ** 2 + 1e-6).sum(-1)


env = GreenLightVecEnv(a.n_envs, uncertainty_scale=a.uncertainty_scale, seed=666)
B, D = a.n_envs, env.obs_dim
rb = DeviceReplayBuffer(env, a.buffer_size, gamma=GAMMA, seed=0)
actor = Actor(D).to(dev)
q1, q2 = mlp(D + NA, 1).to(dev), mlp(D + NA, 1).to(dev)
q1_t, q2_t = copy.deepcopy(q1), copy.deepcopy(q2)
for p in list(q1_t.parameters()) + list(q2_t.parameters()):
    p.requires_grad_(False)
log_alpha = torch.zeros(1, device=dev, requires_grad=True)
opt_pi = torch.optim.Adam(actor.parameters(), lr=a.lr)
opt_q = torch.optim.Adam(list(q1.parameters()) + list(q2.parameters()), lr=a.lr)
opt_a = torch.optim.Adam([log_alpha], lr=a.lr)
target_entropy = -float(NA)


def q_min(n1, n2, obs, act):
    x = torch.cat([obs, act], dim=-1)
    return torch.min(n1(x), n2(x)).squeeze(-1)


def update(batch):
    obs, act, nobs, done, rew = batch.observations, batch.actions, batch.next_observations, batch.dones.squeeze(-1), batch.rewards.squeeze(-1)
    a_pi, logp = actor(obs)
    alpha_loss = -(log_alpha * (logp + target_entropy).detach()).mean()
    opt_a.zero_grad(set_to_none=True)
    alpha_loss.backward()
    opt_a.step()
    alpha = log_alpha.detach().exp()
    with torch.no_grad():
        na, nlogp = actor(nobs)
        target = rew + (1 - done) * GAMMA * (q_min(q1_t, q2_t, nobs, na) - alpha * nlogp)
    x = torch.cat([obs, act], dim=-1)
    q_loss = 0.5 * (F.mse_loss(q1(x).squeeze(-1), target) + F.mse_loss(q2(x).squeeze(-1), target))
    opt_q.zero_grad(set_to_none=True)
    q_loss.backward()
    opt_q.step()
    pi_loss = (alpha * logp - q_min(q1, q2, obs, a_pi)).mean()
    opt_pi.zero_grad(set_to_none=True)
    pi_loss.backward()
    opt_pi.step()
    with torch.no_grad():
        for net, tgt in ((q1, q1_t), (q2, q2_t)):
            for p, pt in zip(net.parameters(), tgt.parameters()):
                pt.lerp_(p, TAU)
    return q_loss, pi_loss


obs = rb.reset()
t_start, env_steps = time.time(), 0
for it in range(a.iters):
    with torch.no_grad():
        if env_steps < a.learning_starts:  # SB3 acts uniformly at random before learning_starts
            act = torch.rand(B, NA, device=dev) * 2 - 1
        else:
            act, _ = actor(obs)
    obs, reward, done = rb.step(act)
    env_steps += B
    q_loss = pi_loss = torch.zeros(())
    if env_steps >= a.learning_starts:
        q_loss, pi_loss = update(rb.sample(a.batch))
    if it % 10 == 9 or it == a.iters - 1:
        torch.cuda.synchronize()
        print(f"iter {it:3d}: mean raw reward {reward.mean().item():+.4f}   buffer {rb.size}/{rb.capacity} slots per env   "
              f"q loss {q_loss.item():.4f}   pi loss {pi_loss.item():+.4f}   alpha {log_alpha.exp().item():.4f}   "
              f"{env_steps / (time.time() - t_start):.3e} env-steps/s incl. updates", flush=True)
rb.close()
env.close()
