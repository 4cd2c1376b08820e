"""bf16-operand emulation of one minibatch of the native PPO update with a STACKED LSTM critic encoder.  TEST INFRASTRUCTURE.

``oracle/ppo_bf16.py:minibatch_grads`` restates the one-layer update; this module restates the same arithmetic for
``nn.LSTM(state_dim, 64, L)`` with L >= 1, built from that module's pieces (its ``r``, ``mlp_forward``, ``mlp_backward``) so that
replacing ``oracle.ppo_bf16.r`` by the identity switches the rounding off here too.  The bf16 rounding points are those of the
one-layer emulation, in every layer: the layer's weights, its input x_t (the states for layer 0, the bf16 h_t of the layer
below above it), its h_t, its saved gates and its gate pre-activation gradients.  The kernels run the layers one after another,
each over all time steps, and back-propagate top layer first: layer k >= 1 also computes dx_t = dgates_t W_ih, which the layer
below adds to the dh of its step t.  For L = 1 the result equals ``oracle.ppo_bf16.minibatch_grads`` exactly.
"""
import math

import torch

import oracle.ppo_bf16 as pb


def minibatch_grads(agent, obs, states, act, old_logp, adv, ret, clip, pi_coef, vf_coef, ent_coef):
    """Gradients of one minibatch the way the native kernels compute them.  Returns ({parameter name: gradient}, stats)."""
    r = pb.r
    with torch.no_grad():
        B = obs.shape[0]
        a_lin, c_lin = pb._linears(agent.actor_mlp), pb._linears(agent.critic_mlp)
        lstm = agent.critic_encoder.layers
        H, T = lstm.hidden_size, states.shape[1]
        # ---- forward
        xs_a, pre = pb.mlp_forward(obs.reshape(B, -1), a_lin)
        mean = torch.tanh(pre)
        xs_in = [r(states[:, t, :]) for t in range(T)]
        layers = []
        for k in range(lstm.num_layers):
            w_ih, w_hh = r(getattr(lstm, f"weight_ih_l{k}")), r(getattr(lstm, f"weight_hh_l{k}"))
            b = getattr(lstm, f"bias_ih_l{k}") + getattr(lstm, f"bias_hh_l{k}")
            b_hi = r(b)
            bias = b_hi + r(b - b_hi)
            h = torch.zeros(B, H, device=obs.device)
            c = torch.zeros(B, H, device=obs.device)
            saved, outs = [], []
            for t in range(T):
                x = xs_in[t]
                g = h @ w_hh.T + x @ w_ih.T + bias
                gi, gf, gg, go = torch.sigmoid(g[:, :H]), torch.sigmoid(g[:, H:2 * H]), torch.tanh(g[:, 2 * H:3 * H]), torch.sigmoid(g[:, 3 * H:])
                c_new = gf * c + gi * gg
                h_new = r(go * torch.tanh(c_new))
                saved.append((h, x, r(gi), r(gf), r(gg), r(go), c, c_new))
                h, c = h_new, c_new
                outs.append(h_new)
            layers.append((w_ih, w_hh, b, saved))
            xs_in = outs
        xs_c, value = pb.mlp_forward(h, c_lin)
        value = value.reshape(B)
        # ---- losses (ppo_asymmetry.py:190-221), as in oracle/ppo_bf16.py
        lsd = 2.0 * agent.log_std
        inv_sd = torch.exp(-lsd)
        z = (act - mean) * inv_sd
        n_act = mean.shape[1]
        logp = -0.5 * (z * z).sum(dim=1) - lsd.sum() - 0.5 * n_act * math.log(2.0 * math.pi)
        log_ratio = logp - old_logp
        ratio = torch.exp(log_ratio)
        s1, s2 = adv * ratio, adv * torch.clamp(ratio, 1.0 - clip, 1.0 + clip)
        dl_dlogp = torch.where(s1 <= s2, -adv * ratio, torch.zeros_like(adv))
        gl = pi_coef * dl_dlogp / B
        dz_a = r(gl.unsqueeze(1) * z * inv_sd * (1.0 - mean * mean))
        dv = value - ret
        dz_c = r((vf_coef * 2.0 * dv / B).unsqueeze(1))
        stats = dict(surrogate=float((-torch.minimum(s1, s2)).mean()), value_loss=float((dv * dv).mean()),
                     kl=float(((ratio - 1.0) - log_ratio).mean()), mean=mean, value=value)
        grads = {"log_std": (gl.unsqueeze(1) * 2.0 * (z * z - 1.0)).sum(dim=0) + ent_coef * -2.0}
        # ---- backward
        ga, _ = pb.mlp_backward(xs_a, a_lin, dz_a)
        for l, (dw, db) in ga.items():
            grads[f"actor_mlp.layers.{2 * l}.weight"], grads[f"actor_mlp.layers.{2 * l}.bias"] = dw, db
        gc, dh_mlp = pb.mlp_backward(xs_c, c_lin, dz_c)
        for l, (dw, db) in gc.items():
            grads[f"critic_mlp.layers.{2 * l}.weight"], grads[f"critic_mlp.layers.{2 * l}.bias"] = dw, db
        dx_above = None                                  # dx_t of the layer above, per step
        for k in range(lstm.num_layers - 1, -1, -1):
            w_ih, w_hh, b, saved = layers[k]
            dh = dh_mlp if k == lstm.num_layers - 1 else torch.zeros(B, H, device=obs.device)
            d_wih, d_whh, d_b = torch.zeros_like(w_ih), torch.zeros_like(w_hh), torch.zeros_like(b)
            dc = torch.zeros(B, H, device=obs.device)
            dxs = [None] * T
            for t in range(T - 1, -1, -1):
                h_prev, x, gi, gf, gg, go, c_prev, c_cur = saved[t]
                if dx_above is not None:
                    dh = dh + dx_above[t]
                tc = torch.tanh(c_cur)
                dc = dc + dh * go * (1.0 - tc * tc)
                dg = r(torch.cat((dc * gg * gi * (1.0 - gi), dc * c_prev * gf * (1.0 - gf), dc * gi * (1.0 - gg * gg), dh * tc * go * (1.0 - go)), dim=1))
                dc = dc * gf
                d_whh += dg.T @ h_prev
                d_wih += dg.T @ x
                d_b += dg.sum(dim=0)
                dh = dg @ w_hh
                if k > 0:
                    dxs[t] = dg @ w_ih
            dx_above = dxs
            grads[f"critic_encoder.layers.weight_ih_l{k}"], grads[f"critic_encoder.layers.weight_hh_l{k}"] = d_wih, d_whh
            grads[f"critic_encoder.layers.bias_ih_l{k}"], grads[f"critic_encoder.layers.bias_hh_l{k}"] = d_b, d_b.clone()
        return grads, stats
