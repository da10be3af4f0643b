"""TEST INFRASTRUCTURE ONLY: a host emulation of the C-ABI entry points the MACBF train step reaches, installed with monkeypatch so that
the PRODUCT's Python (algo/macbf.py, ops.py's autograd Functions, env/base.py, the flat bucket + optimiser glue, native.py's MLP
binding) can be executed in the build container, which has no GPU.  Nothing here is importable from the product, and the product
keeps raising on CPU tensors outside this harness (tests/test_host_cpu.py::test_no_cpu_fallback).

What is emulated, and how:
  * the entry points of csrc/macbf.cu call the HOST BUILD of the very same per-element functions (tests/host_driver/macbf_host.cpp);
  * the rest (edge features, dynamics step, MLP chain, gathers, clip + Adam ...) are restated with torch / the oracle on views
    reconstructed from the raw pointers the product passes, so wrong pointers, pitches, argument orders or shapes show up as
    wrong numbers or crashes.
What this does NOT cover: the CUDA launch code itself and the ctypes signatures (see test_ctypes_signatures_match_the_header).
"""
import ctypes
import math

import numpy as np
import torch

import gcbf_oracle as O

ENV_NAMES = {0: 'SimpleCar', 1: 'DubinsCar', 2: 'SimpleDrone'}
_CT = {torch.float32: ctypes.c_float, torch.float64: ctypes.c_double, torch.int64: ctypes.c_int64, torch.int32: ctypes.c_int32,
       torch.uint8: ctypes.c_uint8}


def T(ptr, rows, ld, cols, dtype=torch.float32):
    """[rows, cols] view (pitch ld) of host memory at `ptr`; writes go to the caller's tensor."""
    if not ptr or rows == 0 or cols == 0:
        return torch.empty(rows, cols, dtype=dtype)
    n = (rows - 1) * ld + cols
    arr = np.ctypeslib.as_array((_CT[dtype] * n).from_address(int(ptr)))
    return torch.as_strided(torch.from_numpy(arr), (rows, cols), (ld, 1))


def V(ptr, n, dtype=torch.float32):
    return T(ptr, 1, n, n, dtype)[0] if n else torch.empty(0, dtype=dtype)


def _addr(byref_obj):
    return ctypes.addressof(byref_obj._obj)


class FakeDevice:
    def __init__(self, host_lib):
        self.host = host_lib
        self.calls = []
        self.step_saved = {}
        self.mlp_saved = {}

    # ---- per-kernel entry points (what _C.call dispatches) ------------------------------------------------------------------
    def gcbf_edge_input_fwd(self, x, node_dim, edge_attr, edge_dim, edge_index, E, out, ld_out):
        if E == 0:
            return
        ei = T(edge_index, 2, E, E, torch.int64)
        num_nodes = int(ei.max()) + 1
        xs, ea = T(x, num_nodes, node_dim, node_dim), T(edge_attr, E, edge_dim, edge_dim)
        T(out, E, ld_out, 2 * node_dim + edge_dim).copy_(torch.cat([xs[ei[1]], xs[ei[0]], ea], dim=1))      # x_i (target), x_j (source), e

    def gcbf_copy2d(self, src, ld_src, dst, ld_dst, rows, cols):
        T(dst, rows, ld_dst, cols).copy_(T(src, rows, ld_src, cols))

    def gcbf_rows_gather(self, src, ld_src, idx, dst, ld_dst, rows, cols):
        ix = V(idx, rows, torch.int64)
        T(dst, rows, ld_dst, cols).copy_(T(src, int(ix.max()) + 1, ld_src, cols)[ix])

    def gcbf_rows_scatter(self, src, ld_src, idx, dst, ld_dst, rows, cols):
        ix = V(idx, rows, torch.int64)
        T(dst, int(ix.max()) + 1, ld_dst, cols)[ix] = T(src, rows, ld_src, cols)

    def gcbf_rowptr_from_targets(self, dst, E, num_nodes, rowptr, flag):
        d = V(dst, E, torch.int64)
        rp = V(rowptr, num_nodes + 1, torch.int32)
        rp.copy_(torch.searchsorted(d.contiguous(), torch.arange(num_nodes + 1)).int())
        bad = E > 0 and (bool((d[1:] < d[:-1]).any()) or int(d.min()) < 0 or int(d.max()) >= num_nodes)
        V(flag, 1, torch.int32)[0] = 1 if bad else 0

    def gcbf_radius_graph_topk_count(self, states, ld, pos_dim, B, N, n, radius, metric, k, rowptr):
        self.host.host_radius_graph_topk(ctypes.c_void_p(states), ld, pos_dim, B, N, n, ctypes.c_float(radius), metric, k,
                                         ctypes.c_void_p(rowptr), None, ctypes.c_int64(0))

    def gcbf_radius_graph_topk_fill(self, states, ld, pos_dim, B, N, n, radius, metric, k, rowptr, edge_index, E):
        if E:
            scratch = torch.zeros(B * n + 1, dtype=torch.int32)
            got = self.host.host_radius_graph_topk(ctypes.c_void_p(states), ld, pos_dim, B, N, n, ctypes.c_float(radius), metric, k,
                                                   ctypes.c_void_p(scratch.data_ptr()), ctypes.c_void_p(edge_index), ctypes.c_int64(E))
            assert got == E and torch.equal(scratch, V(rowptr, B * n + 1, torch.int32))

    def gcbf_edge_masks(self, edge_attr, ld, pos_dim, E, radius, safe, unsafe):
        self.host.host_edge_masks(ctypes.c_void_p(edge_attr), ld, pos_dim, ctypes.c_int64(E), ctypes.c_double(radius), ctypes.c_void_p(safe),
                                  ctypes.c_void_p(unsafe))

    def gcbf_seg_max_fwd(self, msg, ld_msg, rowptr, num_nodes, C, out, ld_out, argmax):
        self.host.host_seg_max_fwd(ctypes.c_void_p(msg), ld_msg, ctypes.c_void_p(rowptr), num_nodes, C, ctypes.c_void_p(out), ld_out,
                                   ctypes.c_void_p(argmax))

    def gcbf_seg_max_bwd(self, d_out, ld_dout, argmax, num_nodes, C, d_msg, ld_dmsg, E):
        self.host.host_seg_max_bwd(ctypes.c_void_p(d_out), ld_dout, ctypes.c_void_p(argmax), num_nodes, C, ctypes.c_void_p(d_msg), ld_dmsg,
                                   ctypes.c_int64(E))

    def gcbf_macbf_loss_partials(self, h, hn, safe, unsafe, E, act, ad, M, alpha, eps, dt, partial):
        f, P = ctypes.c_float, ctypes.c_void_p
        self.host.host_macbf_loss_partials(P(h), P(hn), P(safe), P(unsafe), ctypes.c_int64(E), P(act), ad, ctypes.c_int64(M), f(alpha), f(eps), f(dt),
                                           P(partial))

    def gcbf_macbf_loss_grads(self, h, hn, safe, unsafe, E, act, ad, M, alpha, eps, dt, cu, cs, ch, ca, partial, d_h, d_hn, d_act, scalars):
        f, P = ctypes.c_float, ctypes.c_void_p             # `partial` may have been all-reduced over ranks in between
        self.host.host_macbf_loss_grads(P(h), P(hn), P(safe), P(unsafe), ctypes.c_int64(E), P(act), ad, ctypes.c_int64(M), f(alpha), f(eps), f(dt),
                                        f(cu), f(cs), f(ch), f(ca), P(partial), P(d_h), P(d_hn), P(d_act), P(scalars))

    def gcbf_edge_attr_fwd(self, env, states, ld, edge_index, E, out):
        if E == 0:
            return
        name = ENV_NAMES[env]
        ei = T(edge_index, 2, E, E, torch.int64)
        sd, ed = O.ENV_PARAMS[name]['state_dim'], O.ENV_PARAMS[name]['edge_dim']
        st = T(states, int(ei.max()) + 1, ld, sd)
        T(out, E, ed, ed).copy_(O.edge_attr(name, st, ei))

    def gcbf_edge_attr_bwd(self, env, states, ld, edge_index, E, d_edge_attr, d_states):
        if E == 0:
            return
        name = ENV_NAMES[env]
        ei = T(edge_index, 2, E, E, torch.int64)
        sd, ed = O.ENV_PARAMS[name]['state_dim'], O.ENV_PARAMS[name]['edge_dim']
        rows = int(ei.max()) + 1
        st = T(states, rows, ld, sd).clone().requires_grad_(True)
        with torch.enable_grad():                        # (called from inside an autograd backward: grad mode is off there)
            O.edge_attr(name, st, ei).backward(T(d_edge_attr, E, ed, ed))
        T(d_states, rows, ld, sd).add_(st.grad)

    def _cfg(self, cfg):
        c = cfg._obj
        return ENV_NAMES[c.env], c.num_graphs, c.nodes_per_graph, c.num_agents, c.dt

    def _graph_bits(self, name, B, N, n):
        if name == 'SimpleCar':
            return None
        return torch.cat([torch.ones(n, dtype=torch.bool), torch.zeros(N - n, dtype=torch.bool)]).repeat(B)

    def gcbf_u_ref(self, cfg, states, ld, goal, ldg, K, out):
        name, B, N, n, dt = self._cfg(cfg)
        p = O.ENV_PARAMS[name]
        st = T(states, B * N, ld, p['state_dim'])
        am = self._graph_bits(name, B, N, n)
        g = T(goal, n, ldg, ldg)
        Km = T(K, p['action_dim'], p['state_dim'], p['state_dim']) if K else None
        ag = st if am is None else st[am]
        T(out, B * n, p['action_dim'], p['action_dim']).copy_(torch.cat([O.u_ref(name, ag[b * n:(b + 1) * n], g, Km) for b in range(B)]))

    def _next(self, name, B, N, n, st, act, g, Km, freeze, dt):
        am = self._graph_bits(name, B, N, n)
        p = O.ENV_PARAMS[name]
        outs = []
        for b in range(B):                               # per graph: the oracle's u_ref / reach test take ONE goal set
            s = st[b * N:(b + 1) * N]
            a = act[b * n:(b + 1) * n]
            m = None if am is None else am[:N]
            ag = s if m is None else s[m]
            tot = torch.clamp(a + O.u_ref(name, ag, g, Km), -p['action_lim'], p['action_lim'])
            outs.append(s + O.dynamics(name, s, m, tot, g, bool(freeze) and m is not None) * dt)
        return torch.cat(outs)

    def gcbf_step_fwd(self, cfg, states, ld, action, goal, ldg, K, freeze, nxt, pass_mask):
        name, B, N, n, dt = self._cfg(cfg)
        p = O.ENV_PARAMS[name]
        st = T(states, B * N, ld, p['state_dim']).clone()
        act = T(action, B * n, p['action_dim'], p['action_dim']).clone()
        g = T(goal, n, ldg, ldg).clone()
        Km = T(K, p['action_dim'], p['state_dim'], p['state_dim']).clone() if K else None
        T(nxt, B * N, ld, p['state_dim']).copy_(self._next(name, B, N, n, st, act, g, Km, freeze, dt))
        self.step_saved[int(pass_mask)] = (name, B, N, n, st, act, g, Km, freeze, dt)

    def gcbf_step_bwd(self, cfg, d_next, ld, pass_mask, d_action):
        name, B, N, n, st, act, g, Km, freeze, dt = self.step_saved[int(pass_mask)]
        p = O.ENV_PARAMS[name]
        a = act.clone().requires_grad_(True)
        with torch.enable_grad():
            self._next(name, B, N, n, st, a, g, Km, freeze, dt).backward(T(d_next, B * N, ld, p['state_dim']))
        T(d_action, B * n, p['action_dim'], p['action_dim']).copy_(a.grad)

    def gcbf_grad_sumsq(self, g, count, sumsq):
        V(sumsq, 1, torch.float64)[0] = float((V(g, count).double() ** 2).sum())

    def gcbf_clip_adam(self, p, g, m, v, count, sumsq, max_norm, lr, b1, b2, eps, step):
        P_, G, M_, V_ = V(p, count), V(g, count), V(m, count), V(v, count)
        total = math.sqrt(float(V(sumsq, 1, torch.float64)[0]))
        coef = min(max_norm / (total + 1e-6), 1.0)                      # torch.nn.utils.clip_grad_norm_
        gg = G * coef
        M_.lerp_(gg, 1 - b1)
        V_.mul_(b2).addcmul_(gg, gg, value=1 - b2)
        bc1, bc2 = 1 - b1 ** step, 1 - b2 ** step
        P_.addcdiv_(M_, (V_.sqrt() / math.sqrt(bc2)).add_(eps), value=-lr / bc1)

    # ---- analytic h_dot: the Python-sequenced primal forward (ops.net_forward) + the tangent kernels (host build of jvp_core.h) ------
    def gcbf_linear_fwd(self, X, ldx, W, ldw, bias, inv_sigma, Y, ldy, M, N, K, act, impl, out_amax):
        if M == 0:
            return
        alpha = float(V(inv_sigma, 1)[0]) if inv_sigma else 1.0
        y = alpha * (T(X, M, ldx, K) @ T(W, N, ldw, K).t())
        if bias:
            y = y + V(bias, N)
        y = torch.relu(y) if act == 1 else (torch.tanh(y) if act == 2 else y)
        T(Y, M, ldy, N).copy_(y)

    def gcbf_act_bwd(self, dY, Y, dZ, count, act):
        assert dY and Y and dZ, 'gcbf_act_bwd rejects null pointers even for count 0'
        g, y = V(dY, count), V(Y, count)
        V(dZ, count).copy_(g * (1 - y * y) if act == 2 else (g * (y > 0) if act == 1 else g))

    def gcbf_attn_aggr_fwd(self, msg, ld_msg, gate, rowptr, num_nodes, C, att, aggr, ld_aggr):
        assert C == 256 and ld_msg % 4 == 0 and ld_aggr % 4 == 0
        rp = V(rowptr, num_nodes + 1, torch.int32).long()
        E = int(rp[-1])
        out = T(aggr, num_nodes, ld_aggr, C)
        out.zero_()
        if E == 0:
            return
        dst = torch.repeat_interleave(torch.arange(num_nodes), rp[1:] - rp[:-1])
        a = O.segment_softmax(V(gate, E).reshape(-1, 1).clone(), dst, num_nodes)
        V(att, E).copy_(a.reshape(-1))
        out.copy_(torch.zeros(num_nodes, C).index_add(0, dst, a * T(msg, E, ld_msg, C)))

    def gcbf_sn_power_iter_batched(self, arr, count, ws, ws_floats):
        import torch.nn.functional as F
        for i in range(count):
            a = arr[i]
            W, u, v = T(a.W, a.N, a.ldw, a.K), V(a.u, a.N), V(a.v, a.K)
            v.copy_(F.normalize(torch.mv(W.t(), u), dim=0, eps=1e-12))
            u.copy_(F.normalize(torch.mv(W, v), dim=0, eps=1e-12))
            V(a.inv_sigma, 1)[0] = 1.0 / float(torch.dot(u, torch.mv(W, v)))

    def gcbf_state_dot(self, cfg, states, ld, action, u_ref, goal, ldg, goal_per_graph, freeze, out, ld_out):
        c = cfg._obj
        lim = 2.0 if c.env == 1 else 10.0
        f, P = ctypes.c_float, ctypes.c_void_p
        self.jvp_host.host_state_dot(c.env, c.num_graphs, c.nodes_per_graph, c.num_agents, P(states), ld, P(action), P(u_ref), P(goal), ldg,
                                     c.num_agents if goal_per_graph else 0, f(lim), f(c.speed_limit), f(c.dist2goal), freeze, P(out), ld_out)

    def gcbf_edge_attr_tangent(self, env, states, ld, sdot, ld_sd, edge_index, E, out):
        P = ctypes.c_void_p
        self.jvp_host.host_edge_attr_tangent(env, P(states), ld, P(sdot), ld_sd, P(edge_index), ctypes.c_int64(E), P(out))

    def gcbf_attn_aggr_tangent(self, msg, ld_msg, t_msg, ld_tmsg, att, t_gate, rowptr, num_nodes, C, out, ld_out):
        P = ctypes.c_void_p
        self.jvp_host.host_attn_aggr_tangent(P(msg), ld_msg, P(t_msg), ld_tmsg, P(att), P(t_gate), P(rowptr), num_nodes, C, P(out), ld_out)

    # ---- chain-level MLP (what native.fn(...) returns) ------------------------------------------------------------------------
    def _layers(self, arr, n):
        out = []
        for l in range(n):
            d = arr[l]
            out.append((T(d.W, d.N, d.ldw, d.K), V(d.b, d.N), d.act, d.gW, d.gb, d.ldgw, d.N, d.K))
        return out

    def mlp_forward_workspace_bytes(self, arr, n, rows, save):
        return 4096

    def mlp_backward_workspace_bytes(self, arr, n, rows):
        return 4096

    def mlp_forward(self, arr, n, refresh, x, ldx, rows, out, ld_out, ws, ws_bytes, ctx, stream):
        layers = self._layers(arr, n)
        a = T(x, rows, ldx, layers[0][7]).clone()
        acts = [a]
        for W, b, act, *_ in layers:
            a = torch.nn.functional.linear(a, W, b)
            a = torch.relu(a) if act == 1 else (torch.tanh(a) if act == 2 else a)
            acts.append(a)
        T(out, rows, ld_out, layers[-1][6]).copy_(a)
        if ctx is not None:
            self.mlp_saved[_addr(ctx)] = acts
        self.calls.append('gcbf_mlp_forward')
        return 0

    def mlp_backward(self, arr, n, ctx, d_out, ld_dout, dx, skip_wgrad, ws, ws_bytes, stream):
        layers = self._layers(arr, n)
        acts = self.mlp_saved[_addr(ctx)]
        rows = acts[0].shape[0]
        g = T(d_out, rows, ld_dout, layers[-1][6]).clone()
        for l in range(n - 1, -1, -1):
            W, b, act, gW, gb, ldgw, N, K = layers[l]
            y = acts[l + 1]
            g = g * (y > 0) if act == 1 else (g * (1 - y * y) if act == 2 else g)
            if not skip_wgrad and gW:
                T(gW, N, ldgw, K).add_(g.t() @ acts[l])                # the library ACCUMULATES into the gradient buffers
                V(gb, N).add_(g.sum(0))
            g = g @ W
        if dx:
            T(dx, rows, layers[0][7], layers[0][7]).copy_(g)
        self.calls.append('gcbf_mlp_backward')
        return 0


class _NoStream:
    def wait_event(self, ev):
        pass


class _NoEvent:
    def __init__(self, *a, **k):
        pass

    def record(self, *a, **k):
        pass


def install(monkeypatch, host_lib, jvp_host_lib=None):
    """Route the product's C-ABI calls to a FakeDevice for the duration of a test.  Returns the FakeDevice.  ops and jvp bind `call`
    at import, so both are imported here before anything is patched and their bindings are patched (and restored) as well: a module
    first imported under the patch would otherwise keep the fake for the rest of the session."""
    from gcbf_b200 import _C, jvp, native, ops
    fd = FakeDevice(host_lib)
    fd.jvp_host = jvp_host_lib
    monkeypatch.setattr(torch.cuda, 'Event', _NoEvent)                    # ops.sn_power_iter_batched orders its iterations with events
    monkeypatch.setattr(torch.cuda, 'current_stream', lambda *a, **k: _NoStream())

    def call(name, *args):
        fn = getattr(fd, name, None)
        if fn is None:
            raise AssertionError(f'fake device: {name} is not emulated (the test reached a kernel outside the MACBF step)')
        expected = len(_C._SIGS[name][1]) - 1           # the binding appends the stream
        assert len(args) == expected, f'{name}: {len(args)} arguments, the C prototype has {expected} (+ stream)'
        fd.calls.append(name)
        fn(*args)

    chain = {'gcbf_mlp_forward_workspace_bytes': fd.mlp_forward_workspace_bytes, 'gcbf_mlp_backward_workspace_bytes': fd.mlp_backward_workspace_bytes,
             'gcbf_mlp_forward': fd.mlp_forward, 'gcbf_mlp_backward': fd.mlp_backward, 'gcbf_set_gemm_impl': lambda impl: 0}

    def fn(name):
        if name not in chain:
            raise AssertionError(f'fake device: chain-level entry point {name} is not emulated')
        return chain[name]

    monkeypatch.setattr(_C, 'call', call)
    monkeypatch.setattr(ops, 'call', call)
    monkeypatch.setattr(jvp, 'call', call)
    monkeypatch.setattr(_C, 'require_cuda', lambda *t: None)
    monkeypatch.setattr(_C, 'stream', lambda: None)
    monkeypatch.setattr(native, 'fn', fn)
    monkeypatch.setattr(native, 'workspace', lambda nbytes, device: torch.empty(max(int(nbytes), 256), dtype=torch.uint8))
    return fd
