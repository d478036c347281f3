"""
Policy-in-the-loop rollouts (BASELINE.json configs[4]; SURVEY.md 8f rank 1).

The per-step loop the reference's consumers run on the host -- obs -> network -> clip ->
env.step (/root/reference attic/drl/3dtest.py:36-61) -- stays on the device end to end: the
policy reads the env's observation tensor in place, the step kernel reads the policy's action
tensor in place and writes reward / done straight into row t of the [T, N] rollout buffers
(GAE-ready layout), and the whole T-step horizon is captured once in a CUDA graph and replayed,
so a rollout costs one graph launch instead of T x (policy kernels + 1) launches.

Both rollout classes can also record how each step ended (`store_causes`: the COPTER_CAUSE_* bits,
so that a step-limit truncation is told apart from a termination) and the terminal observation
(`store_final_obs`: with auto-reset, obs of step t + 1 already belongs to the next episode).  `gae`
turns rewards, the learner's values and those records into advantages and returns in one kernel.
"""

import ctypes as C

import torch

from . import _lib
from ._lib import CopterError, VARIANT_IDS


class _EndingRecords:
    """`terminated` / `truncated` [T,N] bool of a rollout that stores its causes: truncated = the env's own step
    limit (CAUSE_TIMEOUT, gymnasium's TimeLimit `truncated`), terminated = any other ending."""

    def _causes(self):
        if self.causes is None:
            raise CopterError('construct the rollout with store_causes=True')
        return self.causes

    @property
    def truncated(self):
        return (self._causes() & _lib.CAUSE_TIMEOUT) != 0

    @property
    def terminated(self):
        c = self._causes()
        return (c != 0) & ((c & _lib.CAUSE_TIMEOUT) == 0)


class PolicyRollout(_EndingRecords):
    """
    env      a CopterVecEnv (already constructed on the target device)
    policy   callable obs[N,O] f32 -> action[N,A] (torch module or function; runs under no_grad)
    horizon  T env.step() calls per rollout
    store_obs  also keep obs_t (the observation the policy saw) in a [T, N, O] buffer
    planar     the policy takes the env's fp32 state planes [3,N,4] in place (see PlanarLinear)
               instead of the packed observation; combine with CopterVecEnv(write_obs=False)
    store_causes     also keep `causes` [T,N] uint8: the COPTER_CAUSE_* bits of the episode that ended
                     on step t, 0 where it goes on (`terminated` / `truncated` are derived from it)
    store_final_obs  also keep `final_obs` [T,N,O] f32: the terminal observation where causes != 0
                     (zero-initialised; rows of steps where nothing ended are left as they were)
    """

    def __init__(self, env, policy, horizon, store_obs=False, use_cuda_graph=True, planar=False,
                 store_causes=False, store_final_obs=False):
        self.env, self.policy, self.horizon = env, policy, int(horizon)
        self.planar = bool(planar)
        if not planar and not env.write_obs:
            raise CopterError('env was built with write_obs=False: use planar=True')
        if planar and store_obs:
            raise CopterError('store_obs needs the packed observation (planar=False)')
        n, dev = env.num_envs, env.device
        self.rewards = torch.zeros((self.horizon, n), dtype=env.dtype, device=dev)
        self.dones = torch.zeros((self.horizon, n), dtype=torch.uint8, device=dev)
        self.obs = torch.zeros((self.horizon, n, env.obs_size), dtype=torch.float32, device=dev) if store_obs else None
        self.causes = torch.zeros((self.horizon, n), dtype=torch.uint8, device=dev) if store_causes else None
        self.final_obs = torch.zeros((self.horizon, n, env.obs_size), dtype=torch.float32, device=dev) if store_final_obs else None
        self.last_obs = env.obs                       # observation after the last step (bootstrap value input)
        self.use_cuda_graph = use_cuda_graph
        self._graph = None
        self.launches_per_rollout = self.horizon      # of OUR kernels; the policy's are torch's

    def _body(self):
        env = self.env
        for t in range(self.horizon):
            if self.obs is not None:
                self.obs[t].copy_(env.obs)
            action = self.policy(env.planar_obs() if self.planar else env.obs)
            if action.dtype != env.dtype:
                action = action.to(env.dtype)
            env.step(action, reward_out=self.rewards[t], done_out=self.dones[t],
                     cause_out=self.causes[t] if self.causes is not None else None,
                     final_obs_out=self.final_obs[t] if self.final_obs is not None else None)

    @torch.no_grad()
    def run(self):
        """One horizon. Returns (rewards [T,N], dones [T,N] bool view, last_obs [N,O])."""
        if not self.env._is_reset:
            raise CopterError('reset() the env before rolling out')
        if not self.use_cuda_graph:
            self._body()
        else:
            if self._graph is None:
                # warm up on a side stream (allocator + lazy module init), roll the env back,
                # then capture
                snapshot = self.env.state_dict()
                s = torch.cuda.Stream(device=self.env.device)
                s.wait_stream(torch.cuda.current_stream(self.env.device))
                with torch.cuda.stream(s):
                    self._body()
                torch.cuda.current_stream(self.env.device).wait_stream(s)
                torch.cuda.synchronize(self.env.device)
                self.env.load_state_dict(snapshot)
                self._graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self._graph):
                    self._body()
            self._graph.replay()
            self.env.launches += self.horizon
        return self.rewards, self.dones.view(torch.bool), self.last_obs


class PlanarLinear(torch.nn.Module):
    """
    First layer of a policy that reads the env's fp32 state planes in place instead of a packed
    [N,O] observation: y = sum_p planes[p][:, :w_p] @ W[:, 4p:4p+w_p].T + b, for the leading
    `obs_size` state components (Lander3D: 10 = planes 0, 1 and half of plane 2).  Same result as
    `linear(obs)` up to summation order; saves the observation write in the step kernel.
    """

    def __init__(self, linear, obs_size):
        super().__init__()
        self.linear, self.obs_size = linear, int(obs_size)

    def forward(self, planes):
        w, out = self.linear.weight, None
        for p in range((self.obs_size + 3) // 4):
            k = min(4, self.obs_size - 4 * p)
            x = planes[p] if k == 4 else planes[p][:, :k]
            y = x.to(w.dtype) @ w[:, 4 * p:4 * p + k].t()
            out = y if out is None else out + y
        return out if self.linear.bias is None else out + self.linear.bias


class FusedMLPPolicy:
    """
    The tanh MLP O -> 64 -> 64 -> A evaluated by ONE hand-written kernel (copter_policy_mlp_strided_f32)
    straight from the env's fp32 state rows -- no observation tensor, no [N,64] intermediates in
    HBM.  Two implementations, 16-bit operands (bf16; fp16 for the hidden layers of the tcgen05 kernel) with fp32
    accumulation in both: tcgen05.mma with the
    accumulators in tensor memory, 128 envs per tile (the default; csrc/copter_policy_tc.cuh), and
    warp-level mma.sync with the activations in registers (csrc/copter_policy.cuh; selected by
    COPTER_B200_POLICY_TC=0 in the environment); FusedPolicyRollout has a fused kernel of each kind.  `net` is a torch.nn.Sequential(Linear, Tanh, Linear, Tanh, Linear,
    Tanh) (e.g. mlp_policy(...).net); its weights are read in place, so optimizer updates to
    fp32 parameters are picked up by the next call.  action = out_offset + out_scale * net(obs).
    Use with PolicyRollout(..., planar=True).
    """

    def __init__(self, env, net, out_scale=1.0, out_offset=0.0):
        lin = [m for m in net if isinstance(m, torch.nn.Linear)]
        if len(lin) != 3 or lin[0].out_features != 64 or lin[1].in_features != 64 or lin[1].out_features != 64 \
                or lin[0].in_features != env.obs_size or lin[2].out_features != env.action_size:
            raise CopterError('FusedMLPPolicy needs Linear(O,64), Linear(64,64), Linear(64,A) with tanh activations')
        if env.dtype != torch.float32:
            raise CopterError('FusedMLPPolicy reads the fp32 state: build the env with dtype=torch.float32')
        self.env, self.lib = env, _lib.load()
        self.params = []
        for m in lin:
            for p in (m.weight, m.bias):
                if p is None or p.dtype != torch.float32 or p.device != env.device or not p.is_contiguous():
                    raise CopterError('policy parameters must be contiguous fp32 tensors (with bias) on the env device')
                self.params.append(p)
        self.out_scale, self.out_offset = float(out_scale), float(out_offset)
        self.action = torch.zeros((env.num_envs, env.action_size), dtype=torch.float32, device=env.device)
        self.launches = 0

    def __call__(self, planes=None):
        env = self.env
        with torch.cuda.device(env.device):
            _lib.check(self.lib.copter_policy_mlp_strided_f32(
                env.state_planes.data_ptr(), *env._state_layout(), env.num_envs, VARIANT_IDS[env.variant], 64,
                *[p.data_ptr() for p in self.params], C.c_float(self.out_scale), C.c_float(self.out_offset),
                self.action.data_ptr(), C.c_void_p(torch.cuda.current_stream(env.device).cuda_stream)),
                'copter_policy_mlp')
        self.launches += 1
        return self.action


class FusedMLPValue:
    """
    The critic Linear(O,64) -> Tanh -> Linear(64,64) -> Tanh -> Linear(64,1) (linear output) evaluated by ONE
    tcgen05 kernel (copter_value_mlp_f32) on fp32 observation rows read in place: a rollout's `obs` / `final_obs`
    [T,N,O], the env's `obs` (a view of its state rows), or any [..., O] tensor whose last dimension has stride 1
    and whose leading dimensions flatten to one stride.  The same rounding as the tcgen05 policy kernel (bf16 rows,
    fp16 hidden activations, fp32 accumulation).  Weights are read in place (fp32), so optimizer updates are seen by
    the next call.

    net             torch.nn.Sequential with those three Linear layers (bias included), fp32, contiguous, on a
                    CUDA device
    variant_or_env  a CopterVecEnv or a variant name: sets O (and the device the parameters must be on)
    """

    def __init__(self, net, variant_or_env):
        if isinstance(variant_or_env, str):
            if variant_or_env not in VARIANT_IDS:
                raise CopterError('unknown variant %r' % (variant_or_env,))
            self.variant, device = variant_or_env, None
        else:
            self.variant, device = variant_or_env.variant, variant_or_env.device
        self.lib = _lib.load()
        self.obs_size = self.lib.copter_obs_size(VARIANT_IDS[self.variant])
        lin = [m for m in net if isinstance(m, torch.nn.Linear)]
        if len(lin) != 3 or lin[0].in_features != self.obs_size or lin[0].out_features != 64 or lin[1].in_features != 64 \
                or lin[1].out_features != 64 or lin[2].in_features != 64 or lin[2].out_features != 1:
            raise CopterError('FusedMLPValue needs Linear(O,64), Linear(64,64), Linear(64,1) with tanh activations')
        if device is None:
            device = lin[0].weight.device
        self.device = torch.device(device)
        self.params = []
        for m in lin:
            for p in (m.weight, m.bias):
                if p is None or p.dtype != torch.float32 or p.device.type != 'cuda' or p.device != self.device \
                        or not p.is_contiguous():
                    raise CopterError('critic parameters must be contiguous fp32 tensors (with bias) on the CUDA device')
                self.params.append(p)
        self.launches = 0

    def __call__(self, rows, select=None, mask=_lib.CAUSE_TIMEOUT, out=None):
        """values [rows.shape[:-1]] fp32.  With `select` (uint8, rows.shape[:-1]) only rows where select & mask != 0
        are evaluated; the other values are left as they were in `out` (zeros when out is None)."""
        O = self.obs_size
        if not isinstance(rows, torch.Tensor) or rows.dtype != torch.float32 or rows.dim() < 1 or rows.shape[-1] != O:
            raise CopterError('rows must be an fp32 tensor [..., %d]' % O)
        if rows.device != self.device:
            raise CopterError('rows must be on the critic device %s' % self.device)
        shape = tuple(rows.shape[:-1])
        if rows.stride(-1) != 1:
            raise CopterError('the last dimension of rows must have stride 1')
        try:
            flat = rows.view(-1, O)
        except RuntimeError:
            raise CopterError('the leading dimensions of rows must flatten to one stride') from None
        m = flat.shape[0]
        stride = flat.stride(0) if m > 1 else O
        if select is not None and (not isinstance(select, torch.Tensor) or select.dtype != torch.uint8
                                   or tuple(select.shape) != shape or select.device != self.device
                                   or not select.is_contiguous()):
            raise CopterError('select must be a contiguous uint8 tensor of shape %s on the critic device' % (shape,))
        if out is None:
            out = (torch.zeros if select is not None else torch.empty)(shape, dtype=torch.float32, device=self.device)
        elif not isinstance(out, torch.Tensor) or out.dtype != torch.float32 or tuple(out.shape) != shape \
                or out.device != self.device or not out.is_contiguous():
            raise CopterError('out must be a contiguous fp32 tensor of shape %s on the critic device' % (shape,))
        with torch.cuda.device(self.device):
            _lib.check(self.lib.copter_value_mlp_f32(
                flat.data_ptr(), stride, m, VARIANT_IDS[self.variant], 64, *[p.data_ptr() for p in self.params],
                select.data_ptr() if select is not None else None, int(mask) & 0xFFFFFFFF, out.data_ptr(),
                C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)), 'copter_value_mlp')
        self.launches += 1
        return out


def policy_log_probs(env, action_std, first_step, horizon, out=None):
    """log N(action; policy(obs), std^2) [T,N] of the actions a FusedPolicyRollout with `action_std` sampled on `env`
    over steps first_step .. first_step + T - 1 (copter_policy_logp_f32): regenerated from the rollout's own noise
    draws, so no network runs and the value is that of the distribution the action was drawn from."""
    if out is None:
        out = torch.empty((int(horizon), env.num_envs), dtype=torch.float32, device=env.device)
    with torch.cuda.device(env.device):
        _lib.check(_lib.load().copter_policy_logp_f32(
            env.seed_value & 0xFFFFFFFFFFFFFFFF, env.env_offset, env.num_envs, int(first_step), int(horizon),
            VARIANT_IDS[env.variant], action_std.data_ptr(), out.data_ptr(),
            C.c_void_p(torch.cuda.current_stream(env.device).cuda_stream)), 'copter_policy_logp')
    return out


class FusedPolicyRollout(_EndingRecords):
    """
    The whole policy-in-the-loop horizon as ONE kernel launch (copter_policy_rollout_f32): every
    warp evaluates the tanh MLP O -> 64 -> 64 -> A for its 32 envs from the state its lanes hold
    in registers and steps them, T times, writing only row t of the [T, N] rollout buffers.
    Step for step identical to PolicyRollout(env, FusedMLPPolicy(env, net, ...), T, planar=True).

    env        a float32 CopterVecEnv with k_substeps == 1
    net        torch.nn.Sequential(Linear(O,64), Tanh, Linear(64,64), Tanh, Linear(64,A), Tanh);
               weights are read in place (fp32), so optimizer updates are seen by the next run()
    horizon    T
    store_obs / store_actions   also record obs_t [T,N,O] (what the policy saw) / action_t [T,N,A]
                                (the command before the env's clip), e.g. for a PPO update
    action_std  None (deterministic policy), a float, or an fp32 CUDA tensor [A] (e.g. exp of a learnable
                log-std, read in place): Gaussian exploration, action = policy(obs) + std * N(0,1), the
                noise from Philox keyed by (seed, global env id, env.rollout_step + t) -- reproducible and
                independent of how the rollout is cut into horizons
    store_causes / store_final_obs   also record `causes` [T,N] uint8 and `final_obs` [T,N,O] as
                PolicyRollout does (the step-limit truncations a learner bootstraps from the value of
                final_obs; `terminated` / `truncated` [T,N] bool are derived from causes)
    critic      None, or the critic torch.nn.Sequential(Linear(O,64), Tanh, Linear(64,64), Tanh, Linear(64,1))
                (fp32, read in place; see FusedMLPValue).  run() then also queues, on the same stream:
                  values [T,N]       the critic on obs (needs store_obs)
                  last_values [N]    the critic on the env's observation after the last step
                  final_values [T,N] the critic on final_obs where the step limit fired, 0 elsewhere
                                     (when store_causes and store_final_obs are set; else None)
    store_log_probs  also record log_probs [T,N]: log N(action; policy(obs), action_std^2) of each sampled
                action, regenerated from the rollout's own noise draws (needs action_std)
    advantages(gamma, lam) is gae() on exactly those buffers (needs a critic and store_causes).
    """

    def __init__(self, env, net, horizon, out_scale=1.0, out_offset=0.0, store_obs=False, store_actions=False,
                 action_std=None, store_causes=False, store_final_obs=False, critic=None, store_log_probs=False):
        probe = FusedMLPPolicy(env, net, out_scale, out_offset)       # same parameter checks
        if env.k_substeps != 1:
            raise CopterError('FusedPolicyRollout steps with k_substeps == 1')
        self.env, self.lib, self.horizon = env, probe.lib, int(horizon)
        if self.horizon < 1:
            raise CopterError('horizon must be >= 1')
        self.params = probe.params
        if action_std is not None and not isinstance(action_std, torch.Tensor):
            action_std = torch.full((env.action_size,), float(action_std), dtype=torch.float32, device=env.device)
        if action_std is not None and (action_std.dtype != torch.float32 or action_std.device != env.device
                                       or action_std.numel() != env.action_size or not action_std.is_contiguous()):
            raise CopterError('action_std must be a contiguous fp32 tensor [A] on the env device')
        self.action_std = action_std
        self.policy = _lib.CopterMlpPolicy(*[p.data_ptr() for p in self.params], 64, float(out_scale), float(out_offset),
                                           action_std.data_ptr() if action_std is not None else None)
        n, dev = env.num_envs, env.device
        self.rewards = torch.zeros((self.horizon, n), dtype=torch.float32, device=dev)
        self.dones = torch.zeros((self.horizon, n), dtype=torch.uint8, device=dev)
        self.obs = torch.zeros((self.horizon, n, env.obs_size), dtype=torch.float32, device=dev) if store_obs else None
        self.actions = torch.zeros((self.horizon, n, env.action_size), dtype=torch.float32, device=dev) if store_actions else None
        self.causes = torch.zeros((self.horizon, n), dtype=torch.uint8, device=dev) if store_causes else None
        self.final_obs = torch.zeros((self.horizon, n, env.obs_size), dtype=torch.float32, device=dev) if store_final_obs else None
        self.critic = self.values = self.last_values = self.final_values = self.log_probs = None
        if critic is not None:
            if not store_obs:
                raise CopterError('a critic needs store_obs=True (the values are those of obs)')
            self.critic = FusedMLPValue(critic, env)
            self.values = torch.zeros((self.horizon, n), dtype=torch.float32, device=dev)
            self.last_values = torch.zeros(n, dtype=torch.float32, device=dev)
            if store_causes and store_final_obs:
                self.final_values = torch.zeros((self.horizon, n), dtype=torch.float32, device=dev)
        if store_log_probs:
            if action_std is None:
                raise CopterError('store_log_probs needs action_std (a deterministic policy has no density)')
            self.log_probs = torch.zeros((self.horizon, n), dtype=torch.float32, device=dev)
        self.launches_per_rollout = 1 + (0 if critic is None else 2 + (self.final_values is not None)) + bool(store_log_probs)

    def run(self):
        """One horizon. Returns (rewards [T,N], dones [T,N] bool view, last_obs [N,O] or None)."""
        env = self.env
        if not env._is_reset:
            raise CopterError('reset() the env before rolling out')
        with torch.cuda.device(env.device):
            b = env._buffers(None, env._force, device=True)
            _lib.check(self.lib.copter_policy_rollout_f32(
                C.byref(env.params), C.byref(b), C.byref(self.policy), env.num_envs, env.env_offset,
                env.seed_value & 0xFFFFFFFFFFFFFFFF, env.rollout_step, self.horizon, VARIANT_IDS[env.variant],
                _lib.F_AUTO_RESET if env.auto_reset else 0, self.rewards.data_ptr(), self.dones.data_ptr(),
                self.actions.data_ptr() if self.actions is not None else None,
                self.obs.data_ptr() if self.obs is not None else None,
                self.causes.data_ptr() if self.causes is not None else None,
                self.final_obs.data_ptr() if self.final_obs is not None else None,
                C.c_void_p(torch.cuda.current_stream(env.device).cuda_stream)), 'copter_policy_rollout')
            first_step = env.rollout_step
            if self.critic is not None:
                self.critic(self.obs, out=self.values)
                self.critic(env.obs, out=self.last_values)
                if self.final_values is not None:
                    self.final_values.zero_()
                    self.critic(self.final_obs, select=self.causes, mask=_lib.CAUSE_TIMEOUT, out=self.final_values)
            if self.log_probs is not None:
                policy_log_probs(env, self.action_std, first_step, self.horizon, out=self.log_probs)
        env.launches += 1
        env.rollout_step += self.horizon
        return self.rewards, self.dones.view(torch.bool), env.obs if env.write_obs else None

    def advantages(self, gamma=0.99, lam=0.95):
        """gae() on this rollout's rewards, values, last_values, causes and final_values: (advantages, returns)
        [T,N].  Without final_values (store_final_obs off) truncations are treated as terminations."""
        if self.critic is None or self.causes is None:
            raise CopterError('advantages() needs a critic and store_causes=True')
        return gae(self.rewards, self.values, self.last_values, self.causes, self.final_values, gamma, lam)


def gae(rewards, values, last_values, causes, final_values=None, gamma=0.99, lam=0.95):
    """
    Generalised advantage estimation on the device (copter_gae_f32, one kernel over the [T,N] rows).
    rewards, values [T,N] f32; last_values [N] f32 (value of the observation after the last step);
    causes [T,N] uint8 (a rollout's `causes`); final_values [T,N] f32 or None (value of `final_obs`,
    read only where a step-limit truncation is).  For t = T-1 .. 0:
        next  = last_values if t == T-1 else values[t+1]
        boot  = next where causes[t] == 0; final_values[t] where the step limit fired (CAUSE_TIMEOUT) and
                final_values is given; 0 otherwise (with final_values None, truncations are terminations)
        delta = rewards[t] + gamma * boot - values[t]
        A[t]  = delta + gamma * lam * (A[t+1] where causes[t] == 0, else 0)
    Returns (advantages [T,N], returns = advantages + values), fp32.  fp32 arithmetic in that order.
    """
    if not all(isinstance(x, torch.Tensor) for x in (rewards, values, last_values, causes)) or \
            (final_values is not None and not isinstance(final_values, torch.Tensor)):
        raise ValueError('gae takes torch tensors')
    if rewards.dim() != 2:
        raise ValueError('rewards must be [T, N], got %s' % (tuple(rewards.shape),))
    T, n = rewards.shape
    if T < 1:
        raise ValueError('gae needs at least one step')
    named = [('rewards', rewards, torch.float32, (T, n)), ('values', values, torch.float32, (T, n)),
             ('last_values', last_values, torch.float32, (n,)), ('causes', causes, torch.uint8, (T, n))]
    if final_values is not None:
        named.append(('final_values', final_values, torch.float32, (T, n)))
    for name, x, dt, shape in named:
        if x.dtype == torch.float64:
            raise ValueError('%s is float64: gae computes in fp32; pass %s.float()' % (name, name))
        if x.dtype != dt:
            raise ValueError('%s must be %s, got %s' % (name, dt, x.dtype))
        if tuple(x.shape) != shape:
            raise ValueError('%s must have shape %s (T, N of rewards), got %s' % (name, shape, tuple(x.shape)))
    for name, x, _, _ in named:
        if x.device.type != 'cuda' or x.device != rewards.device:
            raise CopterError('%s must be on the CUDA device of rewards (there is no CPU fallback)' % name)
        if not x.is_contiguous():
            raise CopterError('%s must be contiguous' % name)
    adv, ret = torch.empty_like(rewards), torch.empty_like(rewards)
    with torch.cuda.device(rewards.device):
        _lib.check(_lib.load().copter_gae_f32(
            rewards.data_ptr(), values.data_ptr(), last_values.data_ptr(), causes.data_ptr(),
            final_values.data_ptr() if final_values is not None else None, n, T, C.c_float(gamma), C.c_float(lam),
            adv.data_ptr(), ret.data_ptr(), C.c_void_p(torch.cuda.current_stream(rewards.device).cuda_stream)),
            'copter_gae')
    return adv, ret


def mlp_policy(obs_size, action_size, hidden=64, dtype=torch.bfloat16, device='cuda', seed=0):
    """The small tanh MLP of SURVEY.md 8d config 5 (O -> 64 -> 64 -> A), random init."""
    g = torch.Generator(device='cpu').manual_seed(seed)
    net = torch.nn.Sequential(
        torch.nn.Linear(obs_size, hidden), torch.nn.Tanh(),
        torch.nn.Linear(hidden, hidden), torch.nn.Tanh(),
        torch.nn.Linear(hidden, action_size), torch.nn.Tanh())
    for p in net.parameters():
        p.data = (torch.randn(p.shape, generator=g) * (0.5 / max(1, p.shape[-1]) ** 0.5))
    net = net.to(device=device, dtype=dtype).eval()

    def policy(obs):
        return net(obs.to(dtype)).float()
    policy.net = net
    return policy
