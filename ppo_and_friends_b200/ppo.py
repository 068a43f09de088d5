"""
The PPO update loop on the B200 path: replaces `PPO._ppo_batch_train` (reference ppo.py:2274-2485)
and the DataLoader / epoch / KL-early-stop section of `PPO.learn` (ppo.py:2178-2238).

`ppo_batch_train(ppo, data_loader, policy_id)` keeps the reference's signature and side effects
(`status_dict[policy_id]["actor loss" | "critic loss" | "kl avg" | "weighted entropy"]`,
`dataset.values` overwritten, value-normaliser statistics advanced on every minibatch), but one
epoch is: draw the permutation with the reference's RNG protocol on the host -> one small prepare
kernel -> a replayed CUDA graph per minibatch (gather + actor/critic forward + fused loss +
backward [+ NCCL all-reduce of the flat gradient] + clip + Adam) -> ONE host sync to read the five
epoch scalars.  Hyper-parameters live in a device block that is refreshed per epoch, so
schedulers keep working without re-capturing.
"""
import ctypes as C
import math
import os
from collections import OrderedDict

import numpy as np
import torch

from . import _lib
from ._lib import HP, ST, check, load, ptr, stream_ptr
from .utils import mpi_utils
from .utils.misc import RunningStatNormalizer


def draw_minibatch_permutation(n):
    """
    The permutation `for batch in DataLoader(dataset, batch_size, shuffle=True)` would use, drawn
    from torch's GLOBAL CPU generator with the same calls in the same order (torch
    utils/data/dataloader.py:705-710 draws the base seed; sampler.py:160-185 draws the seed of a
    private generator and calls randperm) — so minibatch indices are bit-identical to the reference
    for a given `torch.manual_seed` (the CLI seeds rank r with seed + r, ppoaf_cli.py:419).
    """
    _base_seed = torch.empty((), dtype=torch.int64).random_().item()
    seed = int(torch.empty((), dtype=torch.int64).random_().item())
    g = torch.Generator()
    g.manual_seed(seed)
    return torch.randperm(n, generator=g)


class UpdateEngine:
    """Per-policy device state of the fused update (buffers, config structs, captured graphs)."""

    def __init__(self, policy, batch_size, normalize_adv=True, normalize_values=True, value_normalizer=None,
                 use_graphs=None):
        _lib.require_cuda()
        self.policy = policy
        self.device = policy.device
        self.batch_size = int(batch_size)
        self.normalize_adv = bool(normalize_adv)
        self.normalize_values = bool(normalize_values)
        self.value_normalizer = value_normalizer
        self.use_graphs = (os.environ.get("PPOAF_NO_GRAPH", "0") != "1") if use_graphs is None else use_graphs
        # capturing the NCCL all-reduce inside the step graph is opt-in (PPOAF_GRAPH_COLLECTIVE=1)
        self.capture_collective = os.environ.get("PPOAF_GRAPH_COLLECTIVE", "0") == "1"
        # R > 1: gradients are reduced over NVLink peer memory by the fused all-reduce + clip + Adam kernel
        # (PPOAF_PEER=0 falls back to NCCL all-reduce + norm pass + Adam)
        self.peer = None
        self.step_parity = 0
        if mpi_utils.get_num_procs() > 1 and os.environ.get("PPOAF_PEER", "1") != "0" and self.device.type == "cuda":
            from .utils.peer import make_exchange_group
            self.peer = make_exchange_group(policy.nets.n_actor + policy.nets.n_critic, self.device)
        nets = policy.nets
        cfg = _lib.UpdateCfg()
        cfg.actor, cfg.critic = nets.actor.desc, nets.critic.desc
        cfg.head = policy.head
        cfg.act_dim = policy.action_dim
        cfg.use_huber = int(bool(policy.use_huber_loss))
        cfg.normalize_adv = int(self.normalize_adv)
        cfg.normalize_values = int(self.normalize_values)
        cfg.vf_clip_enabled = int(policy.vf_clip is not None)
        cfg.min_std = policy.min_std
        cfg.world_size = mpi_utils.get_num_procs()
        if policy.head == _lib.HEAD_MULTI_CATEGORICAL:
            cfg.section_ends[0], cfg.section_ends[1] = policy.section_ends & 0xFFFFFFFF, policy.section_ends >> 32
        self.cfg = cfg
        dev = self.device
        self.hparams_host = torch.zeros(HP["COUNT"], dtype=torch.float64, pin_memory=True)
        self.hparams = torch.zeros(HP["COUNT"], dtype=torch.float64, device=dev)
        self.epoch_stats = torch.zeros(ST["COUNT"], dtype=torch.float64, device=dev)
        # two pinned slots each for the epoch statistics and the permutation: with KL early stop disabled the trainer keeps
        # one epoch in flight (train_policies), so epoch e + 1 is staged on the host while epoch e still reads its slot
        self._stats_slots = [torch.zeros(ST["COUNT"], dtype=torch.float64, pin_memory=True) for _ in range(2)]
        self._epoch_seq = 0
        self._hp_uploaded = None
        self.mb_cursor = torch.zeros(1, dtype=torch.int32, device=dev)
        ws_bytes = load().ppoaf_update_workspace_bytes(C.byref(cfg), self.batch_size)
        self.workspace = torch.zeros(ws_bytes + 256, dtype=torch.uint8, device=dev)
        # PPOAF_STEP=fused selects the whole-epoch persistent kernel (csrc/fused_step.cu: tcgen05 3xTF32 tiles with A in
        # TMEM, grid barriers instead of launch boundaries).  It is parity-green but measured slower than the launch chain
        # at reference minibatch sizes (DESIGN.md §3.4), so the chain (one CUDA graph of 8 launches per minibatch) stays
        # the default.
        self.fused = (os.environ.get("PPOAF_STEP", "chain") == "fused" and self.peer is None and cfg.world_size == 1
                      and bool(load().ppoaf_ppo_fused_supported(C.byref(cfg))))
        self.fused_workspace = None
        if self.fused:
            fbytes = load().ppoaf_ppo_fused_workspace_bytes(C.byref(cfg), self.batch_size)
            self.fused_workspace = torch.zeros(fbytes + 256, dtype=torch.uint8, device=dev)   # barrier words start at zero
        self.null_state = torch.tensor([0.0, 1.0, 1e-4], dtype=torch.float64, device=dev)
        self._sync_word = torch.zeros(1, dtype=torch.float32, device=dev)
        self._graphs = {}
        self._spec_perm = None          # (n, rng state before, rng state after, permutation) drawn ahead of time
        self._graph_key = None
        self._perm_dev = None
        self.launches_per_step = None

    # -- hyper-parameters (SURVEY row P8: read by the kernels every step) -----------------------------
    def refresh_hparams(self):
        p = self.policy
        # Adam's own hyper-parameters come from the optimizer view (reference: optim.Adam(..., eps=1e-5),
        # policies/ppo_policy.py:341-345), so values restored by load_state_dict are honoured
        g = p.actor_optim.param_groups[0]
        vals = {"LR": float(p.lr()), "ENTROPY_WEIGHT": float(p.entropy_weight()), "SURR_CLIP": float(p.surr_clip),
                "GRAD_CLIP": -1.0 if p.gradient_clip is None else float(p.gradient_clip),
                "KL_WEIGHT": float(p.kl_loss_weight), "VF_CLIP": -1.0 if p.vf_clip is None else float(p.vf_clip),
                "BETA1": float(g["betas"][0]), "BETA2": float(g["betas"][1]), "ADAM_EPS": float(g["eps"]),
                "INV_WORLD": 1.0 / mpi_utils.get_num_procs()}
        if vals == self._hp_uploaded:
            return                       # unchanged since the last upload (also: the pinned staging block is not rewritten
                                         # while an earlier asynchronous copy of it may still be queued)
        h = self.hparams_host
        for k, v in vals.items():
            h[HP[k]] = v
        self.hparams.copy_(h, non_blocking=True)
        self._hp_uploaded = vals

    # -- buffers struct for a given dataset / minibatch size ---------------------------------------------
    def _bufs(self, ds, rows, parity=0, fused=False):
        nets = self.policy.nets
        b = _lib.UpdateBufs()
        b.critic_obs, b.obs = ds.critic_observations.data_ptr(), ds.observations.data_ptr()
        b.raw_actions = ds.raw_actions.data_ptr()
        b.advantages, b.log_probs = ds.advantages.data_ptr(), ds.log_probs.data_ptr()
        b.rewards_to_go, b.values = ds.rewards_to_go.data_ptr(), ds.values.data_ptr()
        b.perm = self._perm_dev.data_ptr()
        b.mb_adv_stats, b.mb_val_stats = self._mb_adv_stats.data_ptr(), self._mb_val_stats.data_ptr()
        grads = self.peer.grads[parity] if self.peer is not None else nets.flat_grads
        b.params, b.grads = nets.flat_params.data_ptr(), grads.data_ptr()
        b.adam_m, b.adam_v, b.adam_step = nets.adam_m.data_ptr(), nets.adam_v.data_ptr(), nets.adam_step.data_ptr()
        b.hparams, b.epoch_stats = self.hparams.data_ptr(), self.epoch_stats.data_ptr()
        b.mb_cursor = self.mb_cursor.data_ptr()
        wst = self.fused_workspace if fused else self.workspace
        ws = wst.data_ptr()
        b.workspace = (ws + 255) // 256 * 256
        b.workspace_bytes = wst.numel() - 256
        b.n_flat = len(ds)
        b.batch, b.batch_size = int(rows), self.batch_size
        if self.peer is not None:                              # push exchange: mirror every gradient store into the peers
            b.n_mirror = len(self.peer.mirror_delta)
            for q, d in enumerate(self.peer.mirror_delta):
                b.mirror_delta[q] = d
        return b

    def _grads(self, bufs):
        check(load().ppoaf_ppo_minibatch_grads(C.byref(self.cfg), C.byref(bufs), stream_ptr()),
              "ppoaf_ppo_minibatch_grads")

    def _apply(self, bufs):
        check(load().ppoaf_ppo_minibatch_apply(C.byref(self.cfg), C.byref(bufs), stream_ptr()),
              "ppoaf_ppo_minibatch_apply")

    def _fused_steps(self, ds, rows, n_steps):
        """n_steps consecutive minibatches of `rows` rows in ONE persistent launch (no graph needed: one launch per epoch)."""
        bufs = self._bufs(ds, rows, fused=True)
        check(load().ppoaf_ppo_fused_steps(C.byref(self.cfg), C.byref(bufs), int(n_steps), stream_ptr()),
              "ppoaf_ppo_fused_steps")

    def _step_eager(self, bufs, parity=0):
        self._grads(bufs)
        if self.peer is not None:
            if bufs.batch > 1:
                self.peer.allreduce_adam(parity, self.policy.nets, self.mb_cursor, self.hparams, stream_ptr())
            else:
                self._apply(bufs)                    # one-row minibatch: only the cursor advances
            return
        if bufs.batch > 1:
            mpi_utils.mpi_avg_gradients(self.policy.nets.flat_grads)
        self._apply(bufs)

    def _ensure_epoch_buffers(self, n):
        n_mb = (n + self.batch_size - 1) // self.batch_size
        dev = self.device
        if self._perm_dev is None or self._perm_dev.numel() != n:
            self._perm_dev = torch.empty(n, dtype=torch.int64, device=dev)
            self._perm_slots = [torch.empty(n, dtype=torch.int64, pin_memory=True) for _ in range(2)]
            self._mb_adv_stats = torch.zeros((n_mb, 2), dtype=torch.float32, device=dev)
            self._mb_val_stats = torch.zeros((n_mb, 2), dtype=torch.float32, device=dev)
            self._mb_val_triples = torch.zeros((n_mb, 3), dtype=torch.float64, device=dev)
            self._graphs.clear()
        return n_mb

    def _ptr_key(self, ds, grads):
        """Every device address a captured step bakes in (ADVICE r1: a key over a subset lets a stale graph replay
        against freed memory when the caching allocator moves only some of the dataset tensors)."""
        nets = self.policy.nets
        return tuple(t.data_ptr() for t in (
            ds.observations, ds.critic_observations, ds.raw_actions, ds.advantages, ds.log_probs, ds.rewards_to_go,
            ds.values, self._perm_dev, self._mb_adv_stats, self._mb_val_stats, grads, nets.flat_params, nets.adam_m,
            nets.adam_v, nets.adam_step, self.hparams, self.epoch_stats, self.mb_cursor, self.workspace)) + (len(ds),)

    def _capture(self, fn):
        graph = torch.cuda.CUDAGraph()
        torch.cuda.synchronize(self.device)
        with torch.cuda.graph(graph):
            fn()
        return graph

    def _launch_step(self, ds, rows):
        parity = self.step_parity if self.peer is not None else 0
        if self.peer is not None and rows > 1:
            self.step_parity ^= 1                      # the peer gradient buffers alternate every real step
            self.policy.nets.flat_grads = self.peer.grads[parity]
        grads = self.peer.grads[parity] if self.peer is not None else self.policy.nets.flat_grads
        key = (rows, parity) + self._ptr_key(ds, grads)
        if not self.use_graphs or rows < 2:
            self._step_eager(self._bufs(ds, rows, parity), parity)
            return
        g = self._graphs.get(key)
        if g is None:
            if len(self._graphs) > 16:
                self._graphs.clear()
            bufs = self._bufs(ds, rows, parity)
            if mpi_utils.get_num_procs() == 1 or self.capture_collective or self.peer is not None:
                g = (self._capture(lambda: self._step_eager(bufs, parity)), None, bufs)
            else:
                # NCCL path: two graphs with the all-reduce of the flat gradient enqueued between them
                g = (self._capture(lambda: self._grads(bufs)), self._capture(lambda: self._apply(bufs)), bufs)
            self._graphs[key] = g
        g[0].replay()
        if g[1] is not None:
            mpi_utils.mpi_avg_gradients(self.policy.nets.flat_grads)
            g[1].replay()

    def _launch_full_minibatches(self, ds, n_full):
        """All full minibatches of an epoch as ONE captured graph: every step is the same chain of launches driven by
        the device-side cursor, so the epoch is n_full copies of it.  Compared with n_full replays of a one-step graph
        this removes the graph-launch gap between steps and lets the programmatic dependencies span step boundaries
        (the first forward GEMM of step k+1 sets up while the optimizer of step k drains)."""
        start = self.step_parity if self.peer is not None else 0
        grads = self.peer.grads[start] if self.peer is not None else self.policy.nets.flat_grads
        key = ("epoch", n_full, start) + self._ptr_key(ds, grads)
        g = self._graphs.get(key)
        if g is None:
            if len(self._graphs) > 16:
                self._graphs.clear()

            def body():
                par = start
                for _ in range(n_full):
                    self._step_eager(self._bufs(ds, self.batch_size, par), par)
                    if self.peer is not None:
                        par ^= 1
            g = (self._capture(body), None, None)
            self._graphs[key] = g
        g[0].replay()
        if self.peer is not None:
            last = start ^ ((n_full - 1) & 1)
            self.step_parity = last ^ 1
            self.policy.nets.flat_grads = self.peer.grads[last]

    # -- the next epoch's permutation, drawn while the GPU is busy --------------------------------------------
    # The draw must consume torch's global CPU generator exactly where the reference's DataLoader would: at the start of
    # the next epoch, and only if that epoch happens (KL early stop, last epoch).  So the generator is rewound after the
    # speculative draw, and the result is used only if the generator is found in exactly that state when the next epoch
    # starts; the generator is then moved to where the draw had left it.
    def _speculate_next_permutation(self, n):
        before = torch.get_rng_state()
        perm = draw_minibatch_permutation(n)
        after = torch.get_rng_state()
        torch.set_rng_state(before)
        self._spec_perm = (n, before, after, perm)

    def _take_speculated_permutation(self, n):
        spec, self._spec_perm = self._spec_perm, None
        if spec is None or spec[0] != n or not torch.equal(torch.get_rng_state(), spec[1]):
            return None
        torch.set_rng_state(spec[2])
        return spec[3]

    # -- one epoch = PPO._ppo_batch_train -------------------------------------------------------------------
    def run_epoch(self, ds):
        """One epoch, synchronously: what `ppo_batch_train` needs (the caller decides about the next epoch from its result)."""
        return self.finish_epoch(self.enqueue_epoch(ds, speculate=True))

    def enqueue_epoch(self, ds, speculate=False):
        """Enqueue one epoch on the current stream and return a token for `finish_epoch`.  Nothing here waits for the GPU:
        the permutation and the statistics travel through pinned slots that alternate from epoch to epoch, so the caller
        may stage the next epoch while this one runs (at most one epoch ahead: two slots)."""
        n = len(ds)
        n_mb = self._ensure_epoch_buffers(n)
        lib = load()
        self.refresh_hparams()
        perm = self._take_speculated_permutation(n)
        if perm is None:
            perm = draw_minibatch_permutation(n)
        slot = self._epoch_seq & 1
        self._epoch_seq += 1
        perm_host = self._perm_slots[slot]
        perm_host.copy_(perm)
        self._perm_dev.copy_(perm_host, non_blocking=True)
        check(lib.ppoaf_epoch_prepare(ptr(self._perm_dev), ptr(ds.advantages), ptr(ds.rewards_to_go), n, self.batch_size,
                                      ptr(self._mb_adv_stats), ptr(self._mb_val_triples), stream_ptr()),
              "ppoaf_epoch_prepare")
        if self.normalize_values:
            triples = mpi_utils.all_gather_cat(self._mb_val_triples).contiguous()     # [R, n_mb, 3]
            state = self.value_normalizer.running_stats.state if self.value_normalizer is not None else self.null_state
            check(lib.ppoaf_value_stats_sequence(ptr(state), ptr(triples), triples.shape[0], n_mb, 1e-8,
                                                 ptr(self._mb_val_stats), stream_ptr()), "ppoaf_value_stats_sequence")
        elif self.peer is not None:
            # no collective precedes the first gradient exchange of this epoch: line the ranks up on the stream, so the
            # spin budget of the in-kernel cross-GPU barrier only has to cover the skew inside one epoch (ADVICE r1)
            mpi_utils.allreduce_sum_(self._sync_word)
        self.epoch_stats.zero_()
        self.mb_cursor.zero_()
        n_full = n // self.batch_size
        # PPOAF_EPOCH_GRAPH=0 falls back to one graph replay per minibatch
        eg = os.environ.get("PPOAF_EPOCH_GRAPH", "1")
        if self.fused:
            rem = n - n_full * self.batch_size
            if n_full >= 1:
                self._fused_steps(ds, self.batch_size, n_full)
            if rem >= 2:
                self._fused_steps(ds, rem, 1)
            elif rem == 1:                                     # the reference skips one-row minibatches: the cursor moves on
                self._apply(self._bufs(ds, 1))
        elif (self.use_graphs and n_full >= 2 and eg == "1"
                and (mpi_utils.get_num_procs() == 1 or self.peer is not None)):
            self._launch_full_minibatches(ds, n_full)          # ONE graph for all full minibatches of the epoch
            if n - n_full * self.batch_size > 0:
                self._launch_step(ds, n - n_full * self.batch_size)
        else:
            for k in range(n_mb):
                rows = min(self.batch_size, n - k * self.batch_size)
                self._launch_step(ds, rows)
        stats_host = self._stats_slots[slot]
        stats_host.copy_(self.epoch_stats, non_blocking=True)
        done = torch.cuda.Event()
        done.record(torch.cuda.current_stream(self.device))
        if speculate:
            self._speculate_next_permutation(n)                         # host work while the GPU runs the epoch
        return (stats_host, done)

    def finish_epoch(self, token):
        stats_host, done = token
        done.synchronize()                                              # the one host wait of the epoch
        return stats_host.clone()


def _get_engine(ppo, policy_id, batch_size):
    policy = ppo.policies[policy_id]
    eng = getattr(policy, "_engine", None)
    vn = ppo.value_normalizers[policy_id] if getattr(ppo, "normalize_values", False) else None
    if (eng is None or eng.batch_size != batch_size or eng.normalize_adv != bool(ppo.normalize_adv)
            or eng.normalize_values != bool(ppo.normalize_values) or eng.value_normalizer is not vn):
        eng = UpdateEngine(policy, batch_size, ppo.normalize_adv, ppo.normalize_values, vn)
        policy._engine = eng
    return eng


def ppo_batch_train(ppo, data_loader, policy_id):
    """
    Drop-in for `PPO._ppo_batch_train(self, data_loader, policy_id)` (ppo.py:2274-2485).
    `data_loader` needs `.dataset` (a built ppo_and_friends_b200 PPODataset) and `.batch_size`.
    """
    policy = ppo.policies[policy_id]
    if policy.frozen:
        return
    ds = data_loader.dataset
    eng = _get_engine(ppo, policy_id, int(data_loader.batch_size))
    _record_epoch(ppo, policy_id, eng, eng.run_epoch(ds).numpy())


def _check_epoch_flags(st):
    if st[ST["BAD_VALUE"]] > 0:
        mpi_utils.abort("ERROR: evaluate value or action prediction contains nan values!")
    if st[ST["BAD_RATIO"]] > 0:
        mpi_utils.abort("ERROR: ratios are nan or inf!")


def _record_epoch(ppo, policy_id, eng, st):
    """Epoch statistics -> status dictionary (ppo.py:2471-2485), one packed all-reduce when R > 1."""
    policy = ppo.policies[policy_id]
    _check_epoch_flags(st)
    peer_err = float(eng.peer.error_flag() != 0) if eng.peer is not None else 0.0
    sums = np.array([st[ST["COUNTER"]], st[ST["ENTROPY"]], st[ST["ACTOR_LOSS"]], st[ST["CRITIC_LOSS"]], st[ST["KL"]], peer_err])
    if mpi_utils.get_num_procs() > 1:                                   # ppo.py:2471-2475, one packed all-reduce
        t = torch.as_tensor(sums).to(policy.device)
        mpi_utils.allreduce_sum_(t)
        sums = t.cpu().numpy()
    if sums[5] > 0:                       # the flag travels with the statistics, so EVERY rank aborts (comm.Abort semantics)
        mpi_utils.abort("ERROR: a rank did not reach the gradient exchange (peer barrier timed out)")
    counter, total_entropy, total_actor, total_critic, total_kl = sums[:5]
    w_entropy = total_entropy * policy.entropy_weight()
    sd = ppo.status_dict[policy_id]
    sd["weighted entropy"] = w_entropy / counter
    sd["actor loss"] = total_actor / counter
    sd["critic loss"] = total_critic / counter
    sd["kl avg"] = total_kl / counter


class _Loader:
    """What the trainer needs from a DataLoader: `.dataset` and `.batch_size`."""

    def __init__(self, dataset, batch_size):
        self.dataset, self.batch_size = dataset, batch_size


def train_policies(ppo):
    """
    The update half of one `PPO.learn` iteration (ppo.py:2178-2238): per policy, up to
    `epochs_per_iter` epochs with optional advantage recalculation and KL early stop, then
    `clear_dataset` is left to the caller exactly where the reference does it.
    Returns {policy_id: epochs actually run}.
    """
    epochs_run = {}
    for policy_id, policy in ppo.policies.items():
        if policy.frozen:
            continue
        loader = _Loader(policy.dataset, ppo.batch_size)
        if _no_early_stop(policy) and ppo.epochs_per_iter > 1 and os.environ.get("PPOAF_PIPELINE_EPOCHS", "1") == "1":
            epochs_run[policy_id] = _train_policy_pipelined(ppo, loader, policy_id)
            continue
        n_ep = 0
        for epoch_idx in range(ppo.epochs_per_iter):
            if epoch_idx > 0 and getattr(ppo, "recalc_advantages", False):
                loader.dataset.recalculate_advantages()
            ppo_batch_train(ppo, loader, policy_id)
            n_ep += 1
            if policy.target_kl is not None and ppo.status_dict[policy_id]["kl avg"] > policy.target_kl:
                if getattr(ppo, "verbose", False):
                    mpi_utils.rank_print("Target KL of {} has been reached. Ending early (after {} epochs)".format(
                        policy.target_kl, epoch_idx + 1))
                break
        epochs_run[policy_id] = n_ep
    return epochs_run


def _no_early_stop(policy):
    """`kl avg > target_kl` (ppo.py:2222-2232) can never hold: no host decision separates two epochs."""
    t = policy.target_kl
    return t is None or (isinstance(t, (int, float)) and math.isinf(t) and t > 0)


def _train_policy_pipelined(ppo, loader, policy_id):
    """
    All epochs of one policy with ONE epoch kept in flight: epoch e + 1 (permutation upload, per-epoch statistics kernels,
    the captured minibatch graph) is enqueued before the host waits for epoch e, so the GPU never idles between epochs.
    Only legal when nothing the host reads from epoch e decides about epoch e + 1, i.e. when KL early stop is disabled
    (`_no_early_stop`); the operations and their order on the stream - and the draws from torch's CPU generator - are exactly
    those of the epoch-by-epoch loop, so the results are bit-identical.  The status dictionary is written once, from the
    last epoch (the reference overwrites it every epoch); the NaN / Inf checks of the earlier epochs run one epoch late.
    """
    policy = ppo.policies[policy_id]
    eng = _get_engine(ppo, policy_id, int(loader.batch_size))
    pending = None
    for epoch_idx in range(ppo.epochs_per_iter):
        if epoch_idx > 0 and getattr(ppo, "recalc_advantages", False):
            loader.dataset.recalculate_advantages()
        token = eng.enqueue_epoch(loader.dataset)
        if pending is not None:
            _check_epoch_flags(eng.finish_epoch(pending).numpy())
        pending = token
    _record_epoch(ppo, policy_id, eng, eng.finish_epoch(pending).numpy())
    return ppo.epochs_per_iter


class PPOUpdateState:
    """
    The slice of the reference `PPO` object the update path reads (ppo.py:126-708): policies, batch
    size, epochs, normalisation switches, value normalisers and the status dict.  A real reference
    `PPO` instance can be passed to `ppo_batch_train` / `train_policies` instead (duck-typed).
    """

    def __init__(self, policies, batch_size=256, epochs_per_iter=10, normalize_adv=True, normalize_values=True,
                 recalc_advantages=False, device="cuda", verbose=False):
        self.policies = OrderedDict(policies)
        self.batch_size, self.epochs_per_iter = batch_size, epochs_per_iter
        self.normalize_adv, self.normalize_values = normalize_adv, normalize_values
        self.recalc_advantages = recalc_advantages
        self.verbose = verbose
        self.device = torch.device(device)
        self.status_dict = OrderedDict({"global status": OrderedDict(iteration=0, timesteps=0)})
        self.value_normalizers = {}
        for pid in self.policies:
            self.status_dict[pid] = OrderedDict()
            if normalize_values:
                self.value_normalizers[pid] = RunningStatNormalizer(pid + "-value_normalizer", self.device)
