"""Thin torch-tensor wrappers over the C ABI (include/usip_b200.h).  PyTorch is used for device
memory and streams only; every computation below happens in libusip_b200.so.  All functions launch on
torch's current CUDA stream and never synchronise."""
import ctypes

import torch

from . import _lib
from ._lib import LayerDesc, check

i32 = torch.int32
f32 = torch.float32


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _req(t, dtype, name):
    if not t.is_cuda:
        raise RuntimeError("%s must be a CUDA tensor/variable" % name)       # index_max.cpp:119-121
    if not t.is_contiguous():
        raise RuntimeError("%s must be contiguous" % name)
    if t.dtype != dtype:
        raise RuntimeError("%s: expected dtype %s, got %s" % (name, dtype, t.dtype))


def tile_rows():
    return _lib.load().usip_layer_tile_rows()


def stat_slots(P, Cout, precision=0, group=0, want_group=False):
    """Rows of the [slots, 2, Cout] BN-statistic partial buffer usip_layer_fwd fills for this layer shape."""
    d = _lib.LayerDesc()
    d.P, d.Cout, d.precision, d.group = int(P), int(Cout), int(precision), int(group)
    d.gmax = 1 if want_group else None          # only tested for NULL-ness by the query
    return _lib.load().usip_layer_stat_slots(ctypes.byref(d))


# ----------------------------------------------------------------------------- reference operators
def index_max(data, index, K):
    """(B,C,N) f32, (B,N) i32 -> (B,C,K) i32.  index_max.forward_cuda_shared_mem semantics."""
    _req(data, f32, "data"); _req(index, i32, "index")
    B, C, N = data.shape
    out = torch.empty((B, C, int(K)), dtype=i32, device=data.device)
    scratch = None
    if K * 12 > 200 * 1024:
        scratch = torch.empty((B * C * K,), dtype=torch.int64, device=data.device)
    with torch.cuda.device(data.device):
        check(_lib.load().usip_index_max_f32(_p(data), _p(index), _p(out), _p(scratch), B, C, N, int(K), _stream()),
              "usip_index_max_f32")
    return out


def ball_query_dist(dist, radius, K):
    _req(dist, f32, "node_to_point_dist")
    B, M, N = dist.shape
    out = torch.empty((B, M, int(K)), dtype=i32, device=dist.device)
    with torch.cuda.device(dist.device):
        check(_lib.load().usip_ball_query_dist_f32(_p(dist), float(radius), _p(out), B, M, N, int(K), _stream()),
              "usip_ball_query_dist_f32")
    return out


_BG_SCRATCH = {}


def _ball_group_scratch(lib, device, B, S, N, M, K):
    """Persistent scratch of the bucket-grid ball query, one per (device, stream, batch): its counter region is cleared once
    here and left cleared by every call (include/usip_b200.h), so the hot path launches no memset."""
    stream = torch.cuda.current_stream()
    key = (device.index, stream.cuda_stream, B)
    ent = _BG_SCRATCH.get(key)
    if ent is None:
        nbytes = int(lib.usip_ball_group_scratch_bytes(B, S, N, M, K))
        buf = torch.empty((max(nbytes, 16),), dtype=torch.uint8, device=device)
        check(lib.usip_ball_group_scratch_init(_p(buf), nbytes, B, _stream()), "usip_ball_group_scratch_init")
        _lib.LAUNCHES[0] -= 1                      # a memset, not one of our kernels
        ent = _BG_SCRATCH[key] = (buf, nbytes)
    return ent


def ball_group(xyz, feat, centers, radius, K, want_group=True, rows_ld=0):
    """Fused distance + ball query + gather + decentre.  Returns (idx (B,M,K) i32, group (B,3+S,M,K) f32)."""
    _req(xyz, f32, "xyz"); _req(centers, f32, "centers")
    B, _, N = xyz.shape
    M = centers.shape[2]
    S = 0 if feat is None else feat.shape[1]
    if S:
        _req(feat, f32, "feat")
    lib = _lib.load()
    idx = torch.empty((B, M, int(K)), dtype=i32, device=xyz.device)
    grp = torch.empty((B, 3 + S, M, int(K)), dtype=f32, device=xyz.device) if want_group else None
    rows = torch.empty((B * M * int(K), rows_ld), dtype=f32, device=xyz.device) if rows_ld else None
    with torch.cuda.device(xyz.device):
        scratch, nbytes = _ball_group_scratch(lib, xyz.device, B, S, N, M, int(K))
        check(lib.usip_ball_group_f32(_p(xyz), _p(feat) if S else None, _p(centers), float(radius), _p(idx), _p(grp),
                                      _p(rows), rows_ld, _p(scratch), int(nbytes), B, S, N, M, int(K), _stream()),
              "usip_ball_group_f32")
    if rows_ld:
        return idx, grp, rows
    return idx, grp


def knn_group(xyz, feat, centers, K, want_group=True, rows_ld=0):
    """K nearest points of every centre + gather + decentre (RPN_Detector_KNN front end, networks.py:556-565).
    Returns (idx (B,M,K) i32 ascending, group (B,3+S,M,K) f32 or None[, rows [B*M*K, rows_ld]])."""
    _req(xyz, f32, "xyz"); _req(centers, f32, "centers")
    B, _, N = xyz.shape
    M = centers.shape[2]
    S = 0 if feat is None else feat.shape[1]
    if S:
        _req(feat, f32, "feat")
    idx = torch.empty((B, M, int(K)), dtype=i32, device=xyz.device)
    grp = torch.empty((B, 3 + S, M, int(K)), dtype=f32, device=xyz.device) if want_group else None
    rows = torch.empty((B * M * int(K), rows_ld), dtype=f32, device=xyz.device) if rows_ld else None
    with torch.cuda.device(xyz.device):
        check(_lib.load().usip_knn_group_f32(_p(xyz), _p(feat) if S else None, _p(centers), _p(idx), _p(grp), _p(rows), rows_ld,
                                             B, S, N, M, int(K), _stream()), "usip_knn_group_f32")
    if rows_ld:
        return idx, grp, rows
    return idx, grp


def fps(pts, start, k, want_nodes=True):
    """Farthest point sampling.  pts (B,Ns,3) f32, start (B,) i32 -> (idx (B,k) i32, nodes (B,3,k) f32 or None)."""
    _req(pts, f32, "pts"); _req(start, i32, "start")
    B, Ns, _ = pts.shape
    idx = torch.empty((B, int(k)), dtype=i32, device=pts.device)
    nodes = torch.empty((B, 3, int(k)), dtype=f32, device=pts.device) if want_nodes else None
    with torch.cuda.device(pts.device):
        check(_lib.load().usip_fps_f32(_p(pts), _p(start), _p(idx), _p(nodes), B, Ns, int(k), _stream()), "usip_fps_f32")
    return idx, nodes


def nms(keypoints, sigmas, radius):
    """keypoints (B,3,M) f32, sigmas (B,M) f32 -> (idx (B,M) i32 kept indices in emission order, -1 padded; count (B,) i32)."""
    _req(keypoints, f32, "keypoints"); _req(sigmas, f32, "sigmas")
    B, _, M = keypoints.shape
    idx = torch.empty((B, M), dtype=i32, device=keypoints.device)
    cnt = torch.empty((B,), dtype=i32, device=keypoints.device)
    with torch.cuda.device(keypoints.device):
        check(_lib.load().usip_nms_f32(_p(keypoints), _p(sigmas), float(radius), _p(idx), _p(cnt), B, M, _stream()), "usip_nms_f32")
    return idx, cnt


def knn_gather(src, idx):
    _req(src, f32, "som_node"); _req(idx, i32, "som_node_knn_I")
    B, C, N = src.shape
    M, K = idx.shape[1], idx.shape[2]
    out = torch.empty((B, C, M, K), dtype=f32, device=src.device)
    check(_lib.load().usip_knn_gather_f32(_p(src), _p(idx), _p(out), B, C, N, M, K, _stream()), "usip_knn_gather_f32")
    return out


# ----------------------------------------------------------------------------- grouping
def som_assign(xyz, node, count=None, method="auto"):
    """Nearest node of every point (som.query_topk, k = 1).  method: "auto" | "brute" | "grid" (identical results): the grid
    path bins the nodes into cells and searches the shells around each point (usip_som_assign_grid_f32)."""
    _req(xyz, f32, "x"); _req(node, f32, "node")
    B, _, N = xyz.shape
    M = node.shape[2]
    min_idx = torch.empty((B, N), dtype=i32, device=xyz.device)
    if count is None:
        count = torch.zeros((B, M), dtype=i32, device=xyz.device)
    lib = _lib.load()
    if method == "grid" or (method == "auto" and 64 <= M <= 1024 and N >= 1024):
        nbytes = int(lib.usip_som_assign_grid_scratch_bytes(B, M))
        scratch = torch.empty(((nbytes + 15) // 16, 4), dtype=i32, device=xyz.device)
        check(lib.usip_som_assign_grid_f32(_p(xyz), _p(node), _p(min_idx), _p(count), _p(scratch), nbytes, B, N, M, _stream()),
              "usip_som_assign_grid_f32")
        return min_idx, count
    check(lib.usip_som_assign_f32(_p(xyz), _p(node), _p(min_idx), _p(count), B, N, M, _stream()),
          "usip_som_assign_f32")
    return min_idx, count


def cluster_sort(min_idx, M):
    B, N = min_idx.shape
    dev = min_idx.device
    seg_off = torch.empty((B, M + 1), dtype=i32, device=dev)
    perm = torch.empty((B, N), dtype=i32, device=dev)
    row_seg = torch.empty((B, N), dtype=i32, device=dev)
    chunks = (N + 255) // 256
    scratch = torch.empty((B * chunks * M,), dtype=i32, device=dev)
    check(_lib.load().usip_cluster_sort(_p(min_idx), _p(seg_off), _p(perm), _p(row_seg), _p(scratch), B, N, M,
                                        _stream()), "usip_cluster_sort")
    return seg_off, perm, row_seg


def cluster_mean_decenter(xyz, feat, seg_off, perm, M, ldx=8):
    B, _, N = xyz.shape
    S = 0 if feat is None else feat.shape[1]
    cmean = torch.empty((B, 3, M), dtype=f32, device=xyz.device)
    x_aug = torch.empty((B * N, ldx), dtype=f32, device=xyz.device)
    check(_lib.load().usip_cluster_mean_decenter(_p(xyz), _p(feat) if S else None, _p(seg_off), _p(perm), _p(cmean),
                                                 _p(x_aug), ldx, B, S, N, M, _stream()), "usip_cluster_mean_decenter")
    return cmean, x_aug


def segmax(X, C, seg_off, perm, B, N, M, out=None, arg=None, want_arg=True):
    ldx = X.stride(0)
    if out is None:
        out = torch.empty((B * M, C), dtype=f32, device=X.device)
    if arg is None and want_arg:
        arg = torch.empty((B * M, C), dtype=i32, device=X.device)
    check(_lib.load().usip_segmax(_p(X), ldx, _p(seg_off), _p(perm), _p(out), out.stride(0), _p(arg), B, N, M, C,
                                  _stream()), "usip_segmax")
    return out, arg


def knn_nodes(pts, K):
    _req(pts, f32, "pts")
    B, _, M = pts.shape
    out = torch.empty((B, M, K), dtype=i32, device=pts.device)
    check(_lib.load().usip_knn_nodes(_p(pts), _p(out), B, M, K, _stream()), "usip_knn_nodes")
    return out


# ----------------------------------------------------------------------------- shared-MLP stack
def layer_fwd(X, W, bias, P, Cin, Cout, ldx=None, ldw=None, in_scale=None, in_shift=None, in_relu=False,
              addend=None, add_index=None, add_group=0, Y=None, ldy=None, stat_partial=None,
              gmax=None, gmin=None, garg_max=None, garg_min=None, group=0, precision=0, tc_ws=None, tc_packed=False, w_transposed=False, debug_flags=0, debug_clocks=None,
              pack_entry=None):
    d = LayerDesc()
    d.X = X.data_ptr(); d.ldx = X.stride(0) if ldx is None else ldx
    d.P = P; d.Cin = Cin; d.Cout = Cout
    d.W = W.data_ptr(); d.ldw = (W.stride(0) if ldw is None else ldw)
    d.w_transposed = 1 if w_transposed else 0
    d.bias = None if bias is None else bias.data_ptr()
    d.in_scale = None if in_scale is None else in_scale.data_ptr()
    d.in_shift = None if in_shift is None else in_shift.data_ptr()
    d.in_relu = 1 if in_relu else 0
    d.addend = None if addend is None else addend.data_ptr()
    d.ld_add = 0 if addend is None else addend.stride(0)
    d.add_index = None if add_index is None else add_index.data_ptr()
    d.add_group = add_group
    d.Y = None if Y is None else Y.data_ptr()
    d.ldy = 0 if Y is None else (Y.stride(0) if ldy is None else ldy)
    d.stat_partial = None if stat_partial is None else stat_partial.data_ptr()
    d.gmax = None if gmax is None else gmax.data_ptr()
    d.gmin = None if gmin is None else gmin.data_ptr()
    d.garg_max = None if garg_max is None else garg_max.data_ptr()
    d.garg_min = None if garg_min is None else garg_min.data_ptr()
    d.group = group
    d.precision = precision
    d.debug_flags = debug_flags
    d.debug_clocks = debug_clocks.data_ptr() if debug_clocks is not None else None
    if precision == 1:
        if tc_ws is None:
            tc_ws = torch.empty((2 * Cin * Cout,), dtype=f32, device=X.device)
        d.tc_workspace = tc_ws.data_ptr(); d.tc_workspace_bytes = tc_ws.numel() * 4
        d.tc_weights_packed = 1 if tc_packed else 0
        if pack_entry is not None and pack_entry.desc is None:
            # remembered for engine.prepack_weights(): the pack of this layer can then join the one-launch re-pack of a
            # train step (the copy keeps W / workspace pointers; the tensors are kept alive next to it)
            pack_entry.desc = LayerDesc.from_buffer_copy(d)
            pack_entry.keep = (W, tc_ws)
    check(_lib.load().usip_layer_fwd(ctypes.byref(d), _stream()),
          "usip_layer_fwd_tc" if (precision == 1 and not tc_packed) else "usip_layer_fwd")


def layer_tc_pack_many(descs):
    arr = (LayerDesc * len(descs))(*descs)
    check(_lib.load().usip_layer_tc_pack_many(arr, len(descs), _stream()), "usip_layer_tc_pack_many")


def bn_finalize(stat_partial, ntiles, count, C, gamma, beta, eps, momentum, running_mean, running_var,
                scale, shift, save_mean=None, save_invstd=None):
    check(_lib.load().usip_bn_finalize(_p(stat_partial), ntiles, int(count), C, _p(gamma), _p(beta), float(eps),
                                       float(momentum), _p(running_mean), _p(running_var), _p(scale), _p(shift),
                                       _p(save_mean), _p(save_invstd), _stream()), "usip_bn_finalize")


def bn_eval_affine(gamma, beta, running_mean, running_var, eps, scale, shift):
    C = gamma.numel()
    check(_lib.load().usip_bn_eval_affine(_p(gamma), _p(beta), _p(running_mean), _p(running_var), float(eps), C,
                                          _p(scale), _p(shift), _stream()), "usip_bn_eval_affine")


def knn_combine(Z, pts, knn_idx, W, ldw, bias, Y, stat_partial, B, M, K, Cout):
    check(_lib.load().usip_knn_combine(_p(Z), Z.stride(0), _p(pts), _p(knn_idx), _p(W), ldw, _p(bias), _p(Y),
                                       Y.stride(0), _p(stat_partial), B, M, K, Cout, _stream()), "usip_knn_combine")


def group_select(gmax, gmin, scale, shift, out, Q, C):
    check(_lib.load().usip_group_select(_p(gmax), _p(gmin), _p(scale), _p(shift), _p(out), out.stride(0), Q, C,
                                        _stream()), "usip_group_select")


def head_finalize(out4, cluster_mean, lb, B, M):
    kp = torch.empty((B, 3, M), dtype=f32, device=out4.device)
    sig = torch.empty((B, M), dtype=f32, device=out4.device)
    check(_lib.load().usip_head_finalize(_p(out4), out4.stride(0), _p(cluster_mean), float(lb), _p(kp), _p(sig), B, M,
                                         _stream()), "usip_head_finalize")
    return kp, sig


def l2norm_to_bcm(X, B, M):
    out = torch.empty((B, X.shape[1], M), dtype=f32, device=X.device)
    check(_lib.load().usip_l2norm_to_bcm(_p(X), X.stride(0), _p(out), None, B, M, X.shape[1], _stream()), "usip_l2norm_to_bcm")
    return out


# ----------------------------------------------------------------------------- backward of the shared-MLP stack
# G / GY are [rows, C] gradients; rows and channels come from their shapes.  "+=" marks outputs accumulated into.
def head_bwd(g_kp, g_sig, out4, B, M):
    G = torch.empty((B * M, 4), dtype=f32, device=out4.device)
    check(_lib.load().usip_head_bwd(_p(g_kp), _p(g_sig), _p(out4), out4.stride(0), _p(G), B, M, _stream()), "usip_head_bwd")
    return G


def wgrad(GY, X, gW, in_scale=None, in_shift=None, in_relu=False, precision=0):
    """gW [Cout, Cin] += GY^T act(X), act = the layer's prologue (folded BN affine, ReLU)."""
    check(_lib.load().usip_wgrad(_p(GY), GY.stride(0), _p(X), X.stride(0), _p(in_scale), _p(in_shift), 1 if in_relu else 0,
                                 _p(gW), gW.stride(0), GY.shape[0], gW.shape[0], gW.shape[1], precision, _stream()), "usip_wgrad")


def colsum(G, out):
    """out [C] += column sums of G."""
    check(_lib.load().usip_colsum(_p(G), G.stride(0), _p(out), G.shape[0], G.shape[1], _stream()), "usip_colsum")


def bn_bwd_reduce(G, Y, scale, shift, mean, invstd, relu):
    P, C = G.shape
    part = torch.empty(((P + 127) // 128, 2, C), dtype=f32, device=G.device)
    check(_lib.load().usip_bn_bwd_reduce(_p(G), G.stride(0), _p(Y), Y.stride(0), _p(scale), _p(shift), _p(mean), _p(invstd),
                                         1 if relu else 0, _p(part), P, C, _stream()), "usip_bn_bwd_reduce")
    return part


def bn_bwd_finalize(part, count, g_gamma, g_beta):
    """g_gamma / g_beta += the BN parameter gradients over `count` rows; returns the constants (c1, c2) of bn_bwd_apply."""
    ntiles, _, C = part.shape
    c1 = torch.empty(C, dtype=f32, device=part.device); c2 = torch.empty(C, dtype=f32, device=part.device)
    check(_lib.load().usip_bn_bwd_finalize(_p(part), ntiles, count, C, _p(g_gamma), _p(g_beta), _p(c1), _p(c2), 1, _stream()),
          "usip_bn_bwd_finalize")
    return c1, c2


def bn_bwd_apply(G, Y, scale, shift, mean, invstd, c1, c2, relu):
    P, C = G.shape
    GY = torch.empty((P, C), dtype=f32, device=G.device)
    check(_lib.load().usip_bn_bwd_apply(_p(G), G.stride(0), _p(Y), Y.stride(0), _p(scale), _p(shift), _p(mean), _p(invstd),
                                        _p(c1), _p(c2), 1 if relu else 0, _p(GY), GY.stride(0), P, C, _stream()),
          "usip_bn_bwd_apply")
    return GY


def groupmax_bwd_select(Gout, gmax, gmin, amax, amin, scale, shift, mean, invstd, with_stats):
    """-> (gz, argsel[, BN-backward partial sums over the selected rows if with_stats, else None]), all [Q, C]-shaped."""
    Q, C = Gout.shape
    gz = torch.empty((Q, C), dtype=f32, device=Gout.device)
    argsel = torch.empty((Q, C), dtype=i32, device=Gout.device)
    part = torch.empty(((Q + 127) // 128, 2, C), dtype=f32, device=Gout.device) if with_stats else None
    check(_lib.load().usip_groupmax_bwd_select(_p(Gout), Gout.stride(0), _p(gmax), _p(gmin), _p(amax), _p(amin), _p(scale),
                                               _p(shift), _p(mean), _p(invstd), _p(gz), _p(argsel), _p(part), Q, C, _stream()),
          "usip_groupmax_bwd_select")
    return gz, argsel, part


def groupmax_scatter_add(G, gsrc, argsel, K):
    """G [Q*K, C]: row argsel[q, c] of group q, column c += gsrc[q, c]."""
    Q, C = gsrc.shape
    check(_lib.load().usip_groupmax_scatter_add(_p(G), G.stride(0), _p(gsrc), _p(argsel), K, Q, C, _stream()),
          "usip_groupmax_scatter_add")


def groupmax_bwd_apply(Y, gz, argsel, scale, mean, invstd, c1, c2, K):
    P, C = Y.shape[0], gz.shape[1]
    GY = torch.empty((P, C), dtype=f32, device=Y.device)
    check(_lib.load().usip_groupmax_bwd_apply(_p(Y), Y.stride(0), _p(gz), _p(argsel), _p(scale), _p(mean), _p(invstd), _p(c1),
                                              _p(c2), _p(GY), GY.stride(0), K, P, C, _stream()), "usip_groupmax_bwd_apply")
    return GY


def group_sum(G, K):
    Q, C = G.shape[0] // K, G.shape[1]
    out = torch.empty((Q, C), dtype=f32, device=G.device)
    check(_lib.load().usip_group_sum(_p(G), G.stride(0), _p(out), out.stride(0), K, Q, C, _stream()), "usip_group_sum")
    return out


def seg_sum(G, seg_off, B, N, M):
    out = torch.empty((B * M, G.shape[1]), dtype=f32, device=G.device)
    check(_lib.load().usip_seg_sum(_p(G), G.stride(0), _p(seg_off), _p(out), out.stride(0), B, N, M, G.shape[1], _stream()),
          "usip_seg_sum")
    return out


def unpool_scatter(G, gp, arg, accumulate):
    """Backward of segmax: G[arg[q, c], c] = gp[q, c], or += with accumulate."""
    check(_lib.load().usip_unpool_scatter(_p(G), G.stride(0), _p(gp), gp.stride(0), _p(arg), gp.shape[0], gp.shape[1],
                                          1 if accumulate else 0, _stream()), "usip_unpool_scatter")


def knn_combine_bwd(GY, pts, knn_idx, GZ, gW, B, M, K):
    """Backward of knn_combine: GZ += GY scattered by neighbour, gW[:, 0:3] += GY^T delta_xyz."""
    check(_lib.load().usip_knn_combine_bwd(_p(GY), GY.stride(0), _p(pts), _p(knn_idx), _p(GZ), GZ.stride(0), _p(gW),
                                           gW.stride(0), B, M, K, GY.shape[1], _stream()), "usip_knn_combine_bwd")


def l2norm_bwd(g, Y, B, M):
    GY = torch.empty((B * M, Y.shape[1]), dtype=f32, device=Y.device)
    check(_lib.load().usip_l2norm_bwd(_p(g.contiguous()), _p(Y), Y.stride(0), _p(GY), GY.stride(0), B, M, Y.shape[1],
                                      _stream()), "usip_l2norm_bwd")
    return GY


# ----------------------------------------------------------------------------- losses
# databases at least this large go through the cell grid (usip_pairwise_min_grid_f32); smaller ones stay brute force
PAIRWISE_MIN_GRID_FROM = 4096


def pairwise_min(a, b, method="auto"):
    """a (B,3,Ma), b (B,3,Nb) -> (min_d (B,Ma) f32, arg (B,Ma) i32).  method: "auto" | "brute" | "grid" (same result)."""
    _req(a, f32, "a"); _req(b, f32, "b")
    B, _, Ma = a.shape
    Nb = b.shape[2]
    d = torch.empty((B, Ma), dtype=f32, device=a.device)
    arg = torch.empty((B, Ma), dtype=i32, device=a.device)
    lib = _lib.load()
    if method == "grid" or (method == "auto" and Nb >= PAIRWISE_MIN_GRID_FROM):
        nbytes = int(lib.usip_pairwise_min_grid_scratch_bytes(B, Nb))
        scratch = torch.empty(((nbytes + 15) // 16, 4), dtype=i32, device=a.device)
        check(lib.usip_pairwise_min_grid_f32(_p(a), _p(b), _p(d), _p(arg), _p(scratch), nbytes, B, Ma, Nb, _stream()),
              "usip_pairwise_min_grid_f32")
        return d, arg
    packed = torch.empty((B, Ma), dtype=torch.int64, device=a.device)
    check(lib.usip_pairwise_min_f32(_p(a), _p(b), _p(d), _p(arg), _p(packed), B, Ma, Nb, _stream()),
          "usip_pairwise_min_f32")
    if Nb <= 2048:
        _lib.LAUNCHES[0] -= 2          # small databases take the single-kernel path (no init / finish launches)
    return d, arg


def pairwise_min_bwd(a, b, d, arg, g, want_b=False, scale=1.0):
    """Gradient of d_i = min_j ||a_i - b_j|| w.r.t. a (and b): g (B,Ma) upstream, times `scale` -> (ga, gb or None)."""
    B, _, Ma = a.shape
    ga = torch.empty_like(a)
    gb = torch.zeros_like(b) if want_b else None
    check(_lib.load().usip_pairwise_min_bwd(_p(a), _p(b), _p(d), _p(arg), _p(g.contiguous()), float(scale), _p(ga), _p(gb),
                                            B, Ma, b.shape[2], _stream()), "usip_pairwise_min_bwd")
    return ga, gb


def chamfer_prob_reduce(d_sd, i_sd, d_ds, i_ds, sig_src, sig_dst):
    B, M = d_sd.shape
    N = d_ds.shape[1]
    out = torch.empty((3,), dtype=f32, device=d_sd.device)
    check(_lib.load().usip_chamfer_prob_reduce(_p(d_sd), _p(i_sd), _p(d_ds), _p(i_ds), _p(sig_src), _p(sig_dst),
                                               _p(out), B, M, N, _stream()), "usip_chamfer_prob_reduce")
    return out


def chamfer_prob_bwd(src, dst, sig_src, sig_dst, d_sd, i_sd, d_ds, i_ds, gout):
    B, _, M = src.shape
    N = dst.shape[2]
    g_src = torch.zeros_like(src); g_dst = torch.zeros_like(dst)
    g_ss = torch.zeros_like(sig_src); g_sd = torch.zeros_like(sig_dst)
    check(_lib.load().usip_chamfer_prob_bwd(_p(src), _p(dst), _p(sig_src), _p(sig_dst), _p(d_sd), _p(i_sd), _p(d_ds), _p(i_ds),
                                            _p(gout), _p(g_src), _p(g_dst), _p(g_ss), _p(g_sd), B, M, N, _stream()),
          "usip_chamfer_prob_bwd")
    return g_src, g_dst, g_ss, g_sd


def transform_points(kp, R, scale, shift):
    B, _, M = kp.shape
    out = torch.empty_like(kp)
    check(_lib.load().usip_transform_points(_p(kp), _p(R), _p(scale), _p(shift), _p(out), B, M, _stream()),
          "usip_transform_points")
    return out


def transform_points_bwd(g, R, scale):
    g = g.contiguous()
    B, _, M = g.shape
    gk = torch.empty_like(g)
    check(_lib.load().usip_transform_points_bwd(_p(g), _p(R), _p(scale), _p(gk), B, M, _stream()), "usip_transform_points_bwd")
    return gk


def mean_scale(d, alpha):
    out = torch.empty((1,), dtype=f32, device=d.device)
    check(_lib.load().usip_mean_scale(_p(d), d.numel(), float(alpha), _p(out), _stream()), "usip_mean_scale")
    return out


def point_on_surface(kp, pc, sn, arg, g=None):
    """-> loss (B,M), or with the upstream gradient g (B,M) the gradient w.r.t. kp (B,3,M) instead."""
    B, _, M = kp.shape
    loss = torch.empty((B, M), dtype=f32, device=kp.device) if g is None else None
    g_kp = None if g is None else torch.empty_like(kp)
    check(_lib.load().usip_point_on_surface(_p(kp), _p(pc), _p(sn), _p(arg), _p(g), _p(loss), _p(g_kp), B, M, pc.shape[2],
                                            sn.shape[1], _stream()), "usip_point_on_surface")
    return loss if g is None else g_kp


def desc_pairmin(a, b):
    """a (B,C,Ma), b (B,C,Nb) -> (min_d (B,Ma) f32, arg (B,Ma) i32)."""
    B, C, Ma = a.shape
    d = torch.empty((B, Ma), dtype=f32, device=a.device)
    arg = torch.empty((B, Ma), dtype=i32, device=a.device)
    check(_lib.load().usip_desc_pairmin_f32(_p(a), _p(b), _p(d), _p(arg), B, C, Ma, b.shape[2], _stream()),
          "usip_desc_pairmin_f32")
    return d, arg


def desc_triplet(dpos, dneg, sigma, gamma, sigma_max):
    B, M = dpos.shape
    loss = torch.empty_like(dpos)
    active = torch.empty((B,), dtype=f32, device=dpos.device)
    check(_lib.load().usip_desc_triplet(_p(dpos), _p(dneg), _p(sigma), float(gamma), float(sigma_max), _p(loss), _p(active),
                                        B, M, _stream()), "usip_desc_triplet")
    return loss, active


def desc_triplet_bwd(anc, pos, neg, dpos, ipos, dneg, ineg, sigma, gamma, sigma_max, g_loss):
    B, C, M = anc.shape
    g_a = torch.zeros_like(anc); g_p = torch.zeros_like(pos); g_n = torch.zeros_like(neg)
    check(_lib.load().usip_desc_triplet_bwd(_p(anc), _p(pos), _p(neg), _p(dpos), _p(ipos), _p(dneg), _p(ineg), _p(sigma),
                                            float(gamma), float(sigma_max), _p(g_loss), _p(g_a), _p(g_p), _p(g_n), B, C, M,
                                            pos.shape[2], neg.shape[2], _stream()), "usip_desc_triplet_bwd")
    return g_a, g_p, g_n


# ----------------------------------------------------------------------------- optimizer
def adam_step(p, g, m, v, lr_dev, step_dev, arrive, beta1, beta2, eps, grad_scale):
    with torch.cuda.device(p.device):
        check(_lib.load().usip_adam_step(_p(p), _p(g), _p(m), _p(v), _p(lr_dev), _p(step_dev), _p(arrive), float(beta1),
                                         float(beta2), float(eps), float(grad_scale), p.numel(), _stream()), "usip_adam_step")


# ----------------------------------------------------------------------------- registration evaluation
def desc_knn(a, b, k, na=None, nb=None, want_dist=False):
    """a (B,C,Ma), b (B,C,Mb) f32, na / nb (B) i32 valid counts or None -> idx (B,Ma,k) i32 (-1 where there is no
    candidate) and, with want_dist, dist (B,Ma,k) f32: the k nearest b columns of every a column, ties to the smaller index."""
    _req(a, f32, "a"); _req(b, f32, "b")
    B, C, Ma = a.shape
    Mb = b.shape[2]
    idx = torch.empty((B, Ma, int(k)), dtype=i32, device=a.device)
    dist = torch.empty((B, Ma, int(k)), dtype=f32, device=a.device) if want_dist else None
    with torch.cuda.device(a.device):
        check(_lib.load().usip_desc_knn_f32(_p(a), _p(b), _p(na), _p(nb), _p(idx), _p(dist), B, C, Ma, Mb, int(k), _stream()),
              "usip_desc_knn_f32")
    return (idx, dist) if want_dist else idx


def corr_build(nn12, Mb, nn21=None, na=None, nb=None):
    """nn12 (B,Ma,k12) i32 anc -> pos indices in [0, Mb), nn21 (B,Mb,k21) i32 pos -> anc or None -> (corr (B,nmax,2) i32,
    count (B) i32): the unique (anc, pos) rows in ascending order (rows past count are -1)."""
    _req(nn12, i32, "nn12")
    B, Ma, k12 = nn12.shape
    Mb, k21 = int(Mb), 0
    if nn21 is not None:
        _req(nn21, i32, "nn21")
        if nn21.shape[:2] != (B, Mb):
            raise RuntimeError("nn21: expected (%d, %d, k), got %s" % (B, Mb, tuple(nn21.shape)))
        k21 = nn21.shape[2]
    nmax = max(1, min(Ma * k12 + Mb * k21, Ma * Mb))
    corr = torch.empty((B, nmax, 2), dtype=i32, device=nn12.device)
    count = torch.empty((B,), dtype=i32, device=nn12.device)
    with torch.cuda.device(nn12.device):
        check(_lib.load().usip_corr_build(_p(nn12), k12, _p(nn21), k21, _p(na), _p(nb), _p(corr), _p(count), B, Ma, Mb, nmax,
                                          _stream()), "usip_corr_build")
    return corr, count


def ransac_rt(anc_xyz, pos_xyz, corr, ncorr, threshold, max_trials, p, seed, samples=None, want_samples=False):
    """Batched RANSAC rigid fit (include/usip_b200.h): anc_xyz (B,Ma,3), pos_xyz (B,Mb,3) f64, corr (B,nmax,2) i32, ncorr (B)
    i32 -> dict of Rt (B,3,4) f64, n_inliers, trialcount, best_trial, status (B) i32, inlier_mask (B,nmax) u8 and, with
    want_samples, samples (B,max_trials+1,3) i32 (-1 for trials never scored)."""
    f64 = torch.float64
    _req(anc_xyz, f64, "anc_xyz"); _req(pos_xyz, f64, "pos_xyz"); _req(corr, i32, "corr"); _req(ncorr, i32, "ncorr")
    B, Ma, _ = anc_xyz.shape
    Mb = pos_xyz.shape[1]
    nmax = corr.shape[1]
    T = int(max_trials) + 1
    dev = anc_xyz.device
    if samples is not None:
        _req(samples, i32, "samples")
        if tuple(samples.shape) != (B, T, 3):
            raise RuntimeError("samples: expected shape %s, got %s" % ((B, T, 3), tuple(samples.shape)))
        n = ncorr.view(B, 1, 1)
        if bool((((samples < 0) | (samples >= n)) & (n > 3)).any()):
            raise RuntimeError("samples: indices must lie in [0, ncorr)")
    out = {"Rt": torch.empty((B, 3, 4), dtype=f64, device=dev),
           "n_inliers": torch.empty((B,), dtype=i32, device=dev), "trialcount": torch.empty((B,), dtype=i32, device=dev),
           "best_trial": torch.empty((B,), dtype=i32, device=dev), "status": torch.empty((B,), dtype=i32, device=dev),
           "inlier_mask": torch.empty((B, nmax), dtype=torch.uint8, device=dev)}
    s_out = torch.full((B, T, 3), -1, dtype=i32, device=dev) if want_samples else None
    lib = _lib.load()
    nbytes = int(lib.usip_ransac_rt_scratch_bytes(B, int(max_trials)))
    scratch = torch.empty(((nbytes + 15) // 16, 2), dtype=f64, device=dev)
    with torch.cuda.device(dev):
        check(lib.usip_ransac_rt(_p(anc_xyz), _p(pos_xyz), _p(corr), _p(ncorr), _p(samples), _p(s_out), float(threshold),
                                 int(max_trials), float(p), int(seed) & 0xFFFFFFFFFFFFFFFF, _p(out["Rt"]), _p(out["n_inliers"]),
                                 _p(out["trialcount"]), _p(out["best_trial"]), _p(out["inlier_mask"]), _p(out["status"]),
                                 _p(scratch), scratch.numel() * 8, B, Ma, Mb, nmax, _stream()), "usip_ransac_rt")
    if want_samples:
        out["samples"] = s_out
    return out
