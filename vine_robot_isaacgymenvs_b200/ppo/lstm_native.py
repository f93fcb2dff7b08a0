"""Host-side orchestration of the kernel-only path for the reference network (MLP -> LSTM 256 -> LayerNorm -> heads):
which kernel runs when, on which buffers.  All arithmetic is in csrc/ (vine_rollout.cu, vine_lstm_net.cu, vine_ppo.cu);
this module only owns the HBM buffers (activation tiles, cell states, gradient workspaces) and issues the launches.

One minibatch (S sequences x L steps, rows ordered [step][sequence]) = 1 MLP forward launch (U tiles), L LSTM steps,
1 head forward/loss/backward, L x (cell backward + backward-data GEMM), 1 MLP backward launch (recompute + weight
gradients), 1 LSTM weight-gradient GEMM, 2 reductions, [all-reduce], [gradient-norm clip over both vectors, with
truncate_grads], 2 Adam launches.
"""
import ctypes as C

import torch

from .. import abi

TB = abi.LSTM_TILE_BYTES // 2        # bf16 elements of one [128 x 128] tile
AB = 128 * 64                        # bf16 elements of one [128 x 64] gate tile


def _ptr(t, off_elems=0):
    return t.data_ptr() + off_elems * t.element_size()


class NativeLstmPath:
    ARENA = True

    def __init__(self, num_obs, seq_len, num_seqs, device, hyper, wgrad_splits=12):
        assert num_seqs % 128 == 0, "sequences per minibatch must be a multiple of the 128-row tile"
        self.lib = abi.load_library()
        self.O, self.L, self.S, self.dev = num_obs, seq_len, num_seqs, device
        self.tiles = num_seqs // 128
        L, S, tl = seq_len, num_seqs, self.tiles
        # every activation / scratch buffer of the path is a view into ONE allocation (ARENA): their relative placement then
        # does not depend on what the caching allocator freed before the agent was built
        elems = lambda s: int(torch.Size(s).numel())  # noqa: E731
        sizes = {"bf": 2 * (elems((L, tl, TB)) + 4 * elems((L, tl, 2, TB)) + 2 * elems((L, tl, 16, AB))),
                 "f32": 4 * (elems((L, S, 256)) + 3 * elems((S, 256)) + elems((L, S, 64)))}
        self._arena = torch.zeros(sizes["bf"] + sizes["f32"] + 64 * 4096, dtype=torch.uint8, device=device) if self.ARENA else None
        self._arena_off = 0

        def alloc(shape, dtype):
            if self._arena is None:
                return torch.zeros(*shape, dtype=dtype, device=device)
            nbytes = elems(shape) * torch.empty(0, dtype=dtype).element_size()
            off = self._arena_off
            self._arena_off = (off + nbytes + 4095) & ~4095
            assert self._arena_off <= self._arena.numel()
            return self._arena[off:off + nbytes].view(dtype).view(*shape)
        bf = lambda *s: alloc(s, torch.bfloat16)  # noqa: E731
        f32 = lambda *s: alloc(s, torch.float32)  # noqa: E731
        self.U, self.HM, self.HH = bf(L, tl, TB), bf(L, tl, 2, TB), bf(L, tl, 2, TB)
        self.ACT, self.DG = bf(L, tl, 16, AB), bf(L, tl, 16, AB)
        self.DH, self.DHREC = bf(L, tl, 2, TB), bf(L, tl, 2, TB)
        self.Cs, self.C0 = f32(L, S, 256), f32(S, 256)
        self.DC = [f32(S, 256), f32(S, 256)]
        self.DH3 = f32(L, S, 64)
        self.head_grads = torch.zeros(abi.LSTM_HEAD_GRAD_PARTS + 1, abi.LSTM_HEAD_GRAD_FLOATS, device=device)   # + 1 row: their sum
        self.splits = min(wgrad_splits, L * tl)
        self.wg_ws = torch.zeros(self.splits, abi.LSTM_WGRAD_BLOCK_FLOATS, device=device)
        self.mlp_ctas = self.lib.vine_ppo_max_ctas()
        self.mlp_ws = torch.empty(self.mlp_ctas, abi.PPO_WS_FLOATS, device=device)
        self.P_mlp, self.P_lstm = self.lib.vine_ppo_num_params(num_obs), self.lib.vine_lstm_num_params(num_obs)
        # both gradient vectors (+ 4 loss statistics each) in ONE buffer: one all-reduce per minibatch across ranks
        self.flat_g = torch.zeros(self.P_mlp + 4 + self.P_lstm + 4, device=device)
        self.flat_g_mlp, self.flat_g_lstm = self.flat_g[:self.P_mlp + 4], self.flat_g[self.P_mlp + 4:]
        self.hyper = hyper
        self._stream = lambda: C.c_void_p(torch.cuda.current_stream(device).cuda_stream)

    # ------------------------------------------------------------------ forward + backward of one minibatch
    def gradients(self, packed_mlp, packed_lstm, obs, scalars, not_done, obs_mean, obs_inv_std, value_stats, logstd, logstd_old,
                  state, debug_out=None, writeback=None, p2p=(None, None), position=(0, 0)):
        """obs f32 [L, S, O], scalars f32 [L, S, 8], not_done f32 [L, S]; self.HM[0] (masked initial hidden state tiles) and
        self.C0 must already hold the initial LSTM state.  Leaves the gradients in flat_g_mlp / flat_g_lstm.
        ``writeback`` = (scalars_src [T, N, 8], seq_len, chunks, num_envs, env_begin, env_count): rl_games'
        dataset.update_mu_sigma -- this pass's mu goes back into the source rows and ``logstd_old`` receives ``logstd``.
        ``p2p`` = (MLP channel, LSTM channel) device pointers: multi-GPU, the two gradient sums go into this rank's peer-visible
        buffers instead of flat_g_* (distributed.P2PChannel).  ``position`` = (mini-epoch, minibatch slot) of this minibatch
        in the iteration: what the learning-rate schedule of vine_ppo_minibatch needs to know, passed to hyper["schedule"]
        (PPOAgent._schedule_fields); without that entry the launch runs the adaptive legacy schedule."""
        lib, L, S, tl, st = self.lib, self.L, self.S, self.tiles, self._stream()
        n = L * S
        act = abi.VinePolicyAct(packed=_ptr(packed_mlp), obs=_ptr(obs), obs_mean=_ptr(obs_mean), obs_inv_std=_ptr(obs_inv_std),
                                value_stats=_ptr(value_stats), n=n, num_obs=self.O, u_out=_ptr(self.U))
        assert lib.vine_policy_act(C.byref(act), st) == 0
        for t in range(L):
            last = t == L - 1
            a = abi.VineLstmStep(params=_ptr(packed_lstm), u=_ptr(self.U[t]), hm=_ptr(self.HM[t]),
                                 c_prev=_ptr(self.Cs[t - 1] if t else self.C0), not_done=_ptr(not_done[t]),
                                 not_done_next=None if last else _ptr(not_done[t + 1]), c=_ptr(self.Cs[t]), hh=_ptr(self.HH[t]),
                                 hm_next=None if last else _ptr(self.HM[t + 1]), act=_ptr(self.ACT[t]), n=S)
            assert lib.vine_lstm_step(C.byref(a), st) == 0
        h = self.hyper
        ht = abi.VineLstmHeadTrain(params=_ptr(packed_lstm), hh=_ptr(self.HH), scalars=_ptr(scalars), logstd=_ptr(logstd),
                                   logstd_old=_ptr(logstd_old), dh=_ptr(self.DH), grads=_ptr(self.head_grads),
                                   debug_out=_ptr(debug_out) if debug_out is not None else None, n=n, inv_B=1.0 / n,
                                   e_clip=h["e_clip"], critic_coef=h["critic_coef"], entropy_coef=h["entropy_coef"],
                                   bounds_loss_coef=h["bounds_loss_coef"], value_loss_unclipped=int(not h.get("clip_value", True)))
        if writeback is not None:
            src, wl, wc, wn, wb, we = writeback
            ht.mu_writeback, ht.wb_seq_len, ht.wb_chunks, ht.wb_num_envs, ht.wb_env_begin, ht.wb_env_count = _ptr(src), wl, wc, wn, wb, we
        hparts = lib.vine_lstm_head_train(C.byref(ht), st)
        assert hparts > 0, hparts
        for t in range(L - 1, -1, -1):
            last = t == L - 1
            cb = abi.VineLstmCellBwd(act=_ptr(self.ACT[t]), c_prev=_ptr(self.Cs[t - 1] if t else self.C0), c=_ptr(self.Cs[t]),
                                     not_done=_ptr(not_done[t]), dh=_ptr(self.DH[t]), dh_rec=None if last else _ptr(self.DHREC[t]),
                                     dc_next=None if last else _ptr(self.DC[(t + 1) & 1]), dg=_ptr(self.DG[t]),
                                     dc_prev=_ptr(self.DC[t & 1]), n=S)
            assert lib.vine_lstm_cell_bwd_tiles(C.byref(cb), st) == 0
            bg = abi.VineLstmBwdGemm(params=_ptr(packed_lstm), dg=_ptr(self.DG[t]), not_done=_ptr(not_done[t]), dh3=_ptr(self.DH3[t]),
                                     dh_rec=_ptr(self.DHREC[t - 1]) if t else None, n=S)
            assert lib.vine_lstm_bwd_gemm(C.byref(bg), st) == 0
        sched = h["schedule"](*position) if "schedule" in h else dict(
            adaptive_lr=int(h.get("adaptive_lr", 1)), kl_threshold=h.get("kl_threshold", 0.008), lr_min=1e-6, lr_max=1e-2)
        mb = abi.VinePpoMinibatch(packed=_ptr(packed_mlp), obs=_ptr(obs), obs_mean=_ptr(obs_mean), obs_inv_std=_ptr(obs_inv_std),
                                  logstd=_ptr(logstd), logstd_old=_ptr(logstd_old), workspace=_ptr(self.mlp_ws), state=_ptr(state),
                                  horizon=1, num_envs=n, env_begin=0, env_count=n, num_obs=self.O, workspace_ctas=self.mlp_ctas,
                                  e_clip=h["e_clip"], critic_coef=h["critic_coef"], entropy_coef=h["entropy_coef"],
                                  bounds_loss_coef=h["bounds_loss_coef"], dh3_ext=_ptr(self.DH3), **sched)
        n_part = lib.vine_ppo_minibatch(C.byref(mb), st)
        assert n_part > 0, n_part
        wb = writeback is not None   # sigma half of update_mu_sigma: after the last reader of logstd_old, before Adam
        assert lib.vine_ppo_reduce(C.c_void_p(_ptr(self.mlp_ws)), n_part, self.O, C.c_void_p(_ptr(self.flat_g_mlp)),
                                   C.c_void_p(_ptr(logstd)) if wb else None, C.c_void_p(_ptr(logstd_old)) if wb else None, p2p[0], st) == 0
        wg = abi.VineLstmWgrad(u=_ptr(self.U), hm=_ptr(self.HM), dg=_ptr(self.DG), workspace=_ptr(self.wg_ws), ntiles=L * tl,
                               splits=self.splits)
        assert lib.vine_lstm_wgrad(C.byref(wg), st) == 0
        assert lib.vine_lstm_reduce(C.c_void_p(_ptr(self.wg_ws)), self.splits, C.c_void_p(_ptr(self.head_grads)), hparts, self.O,
                                    C.c_void_p(_ptr(self.flat_g_lstm)), p2p[1], st) == 0
