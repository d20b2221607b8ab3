// Native (C++) stage drivers: the KPConv-FPN backbone and the geometric transformer as ONE C-ABI call each.
//
// The per-op entry points of geob200.h are the drop-in boundary and what the parity tests call; driven from Python they
// cost ~10 us of host time per op and a pair needs ~340 of them, which makes the host the bottleneck once the kernels are
// fast.  These drivers issue exactly the same kernel sequence as geotransformer_b200/backbone.py and
// geotransformer_b200/modules/transformer/modules.py (bitwise-identical results, tests/test_gpu_native.py) from C++,
// ~2-3 us per launch, with all intermediates in a caller-provided arena.
//
// Reference: experiments/*/backbone.py (KPConvFPN.forward), geotransformer/modules/kpconv/modules.py:107-225,
//            geotransformer/modules/geotransformer/geotransformer.py:114-155,
//            geotransformer/modules/transformer/conditional_transformer.py:97-117.
#include "common.cuh"
#include "geob200.h"

namespace geob200 {

struct Ctx {
    Arena ar;
    void* gn_ws;
    size_t gn_ws_bytes;
    void* stream;
    int groups;
    Ctx(void* p, size_t n) : ar(p, n) {}
    float* fl(int64_t rows, int64_t ch) { return ar.take<float>((size_t)rows * (size_t)ch); }
};

#define TRY(expr)                  \
    do {                           \
        int _rc = (expr);          \
        if (_rc != 0) return _rc;  \
    } while (0)

static int run_kpconv(Ctx& c, const geob200_kpconv_t& k, const float* s_feats, const float* q_pts, const float* s_pts,
                      const int64_t* nbr, int64_t m, int64_t ns, int64_t h, float* out) {
    const bool tc = (k.c_in % 32 == 0) && (k.c_out % 16 == 0) && k.c_out >= 32 && (k.c_out <= 128 || k.c_out % 128 == 0) && m >= 64 &&
                    k.weights_t != nullptr;
    if (tc) {
        const size_t wb = geob200_kpconv_tc_workspace_bytes(m, ns, k.c_in);
        const size_t mark = c.ar.off;
        void* ws = c.ar.take<char>(wb);
        GEOB_REQUIRE(c.ar.ok(), "native: arena too small (kpconv)");
        TRY(geob200_kpconv_tc(s_feats, q_pts, s_pts, nbr, m, ns, h, k.kernel_points, 15, k.weights_t, k.bias, k.c_in, k.c_out, k.sigma,
                              out, ws, wb, c.stream));
        c.ar.off = mark;     // stream-ordered reuse: the next kernel that touches this scratch runs after the GEMM
        return 0;
    }
    const size_t wb = geob200_kpconv_workspace_bytes(ns);
    const size_t mark = c.ar.off;
    void* ws = c.ar.take<char>(wb);
    GEOB_REQUIRE(c.ar.ok(), "native: arena too small (kpconv)");
    TRY(geob200_kpconv(s_feats, q_pts, s_pts, nbr, m, ns, h, k.kernel_points, 15, k.weights, k.bias, k.c_in, k.c_out, k.sigma, out, ws,
                       wb, c.stream));
    c.ar.off = mark;
    return 0;
}

// KPConv -> GroupNorm -> LeakyReLU (ConvBlock / conv part of ResidualBlock); out = normalised activations
static int run_kpconv_norm(Ctx& c, const geob200_kpconv_t& k, const geob200_norm_t& n, const float* s_feats, const float* q_pts,
                           const float* s_pts, const int64_t* nbr, int64_t m, int64_t ns, int64_t h, float* out, const GnSeg& seg) {
    float* y = c.fl(m, k.c_out);
    GEOB_REQUIRE(c.ar.ok(), "native: arena too small (kpconv output)");
    const bool tc = (k.c_in % 32 == 0) && (k.c_out % 16 == 0) && k.c_out >= 32 && (k.c_out <= 128 || k.c_out % 128 == 0) && m >= 64 &&
                    k.weights_t != nullptr;
    if (tc) {
        const size_t wb = geob200_kpconv_tc_workspace_bytes(m, ns, k.c_in);
        const size_t mark = c.ar.off;
        void* ws = c.ar.take<char>(wb);
        GEOB_REQUIRE(c.ar.ok(), "native: arena too small (kpconv)");
        TRY(kpconv_group_norm_impl(s_feats, q_pts, s_pts, nbr, m, ns, h, k.kernel_points, 15, k.weights_t, k.bias, k.c_in, k.c_out,
                                   k.sigma, c.groups, n.gamma, n.beta, 1e-5f, 1, 0.1f, y, out, c.gn_ws, c.gn_ws_bytes, ws, wb, c.stream, seg));
        c.ar.off = mark;     // stream-ordered reuse: the next kernel that touches this scratch runs after the GEMM
        return 0;
    }
    TRY(run_kpconv(c, k, s_feats, q_pts, s_pts, nbr, m, ns, h, y));
    return group_norm_impl(y, m, k.c_out, c.groups, n.gamma, n.beta, 1e-5f, nullptr, 1, 0.1f, out, c.gn_ws, c.gn_ws_bytes, c.stream, seg);
}

// Linear -> GroupNorm (+ residual) (+ LeakyReLU)
static int run_unary(Ctx& c, const geob200_linear_t& l, const geob200_norm_t& n, const float* x, int64_t rows, const float* residual,
                     int leaky, float* out, const GnSeg& seg) {
    float* t = c.fl(rows, l.c_out);
    GEOB_REQUIRE(c.ar.ok(), "native: arena too small (unary)");
    TRY(linear_group_norm_impl(x, l.c_in, l.weight, l.bias, rows, l.c_out, l.c_in, c.groups, n.gamma, n.beta, 1e-5f, residual, leaky,
                               0.1f, t, out, c.gn_ws, c.gn_ws_bytes, c.stream, seg));
    return 0;
}

static int run_resblock(Ctx& c, const geob200_resblock_t& b, const float* feats, int64_t ns, const float* q_pts, const float* s_pts,
                        const int64_t* nbr, int64_t m, int64_t h, float* out, const GnSeg& seg_s, const GnSeg& seg_q,
                        const int* cloud_max = nullptr) {
    const float* x = feats;
    if (b.has_unary1) {
        float* u = c.fl(ns, b.unary1.c_out);
        TRY(run_unary(c, b.unary1, b.norm1, feats, ns, nullptr, 1, u, seg_s));
        x = u;
    }
    float* yn = c.fl(m, b.conv.c_out);
    GEOB_REQUIRE(c.ar.ok(), "native: arena too small (resblock)");
    TRY(run_kpconv_norm(c, b.conv, b.norm_conv, x, q_pts, s_pts, nbr, m, ns, h, yn, seg_q));
    const float* sc = feats;
    if (b.strided) {
        float* mp = c.fl(m, b.c_in);
        GEOB_REQUIRE(c.ar.ok(), "native: arena too small (maxpool)");
        if (cloud_max != nullptr) {
            TRY(maxpool_seg(feats, nbr, m, ns, h, b.c_in, mp, &seg_q, cloud_max, c.stream));
        } else {
            TRY(geob200_maxpool(feats, nbr, m, ns, h, b.c_in, mp, c.stream));
        }
        sc = mp;
    }
    if (b.has_shortcut) {
        float* s2 = c.fl(m, b.shortcut.c_out);
        TRY(run_unary(c, b.shortcut, b.norm_sc, sc, m, nullptr, 0, s2, seg_q));
        sc = s2;
    }
    return run_unary(c, b.unary2, b.norm2, yn, m, sc, 1, out, seg_q);   // leaky(norm(unary2(x)) + shortcut)
}

}  // namespace geob200

using namespace geob200;

extern "C" {

size_t geob200_backbone_workspace_bytes(const geob200_backbone_t* net, const int64_t* level_rows) {
    // generous bound: every block keeps <= 6 activations of its widest channel count, plus the tensor-core KPConv scratch
    size_t total = 1 << 20;
    for (int l = 0; l < net->num_stages; ++l) {
        const size_t rows = (size_t)level_rows[l];
        const size_t ch = (size_t)net->init_dim << (l + 1);
        total += rows * ch * 4 * 24;
        total += geob200_kpconv_tc_workspace_bytes(level_rows[l], l > 0 ? level_rows[l - 1] : level_rows[l], (int64_t)(ch / 2)) + 4096;
    }
    return total;
}

int geob200_backbone_forward(const geob200_backbone_t* net, const float* feats, const float* const* points, const int64_t* level_rows,
                             const int64_t* const* neighbors, const int64_t* neighbor_width, const int64_t* const* subsampling,
                             const int64_t* subsampling_width, const int64_t* const* upsampling, const int64_t* upsampling_width,
                             float* const* out_feats /* [num_stages - finest_decoder + 1], coarse first */, void* gn_workspace,
                             size_t gn_workspace_bytes, void* workspace, size_t workspace_bytes, void* stream) {
    return geob200_backbone_forward_batched(net, feats, points, level_rows, neighbors, neighbor_width, subsampling, subsampling_width,
                                            upsampling, upsampling_width, out_feats, gn_workspace, gn_workspace_bytes, workspace,
                                            workspace_bytes, stream, 1, nullptr, nullptr);
}

size_t geob200_backbone_gn_workspace_bytes(const geob200_backbone_t* net, const int64_t* level_rows, int64_t n_pairs) {
    // the finest level has the most rows, the coarsest encoder output the most channels
    return geob200_group_norm_workspace_bytes(level_rows[0], (int64_t)net->init_dim << net->num_stages, net->groups, n_pairs);
}

int geob200_backbone_forward_batched(const geob200_backbone_t* net, const float* feats, const float* const* points,
                                     const int64_t* level_rows, const int64_t* const* neighbors, const int64_t* neighbor_width,
                                     const int64_t* const* subsampling, const int64_t* subsampling_width,
                                     const int64_t* const* upsampling, const int64_t* upsampling_width, float* const* out_feats,
                                     void* gn_workspace, size_t gn_workspace_bytes, void* workspace, size_t workspace_bytes, void* stream,
                                     int64_t n_pairs, const int64_t* const* cloud_rows_h, const int32_t* const* sub_cloud_max) {
    GEOB_REQUIRE(n_pairs == 1 || sub_cloud_max != nullptr, "backbone: batched execution needs the per-cloud subsampling widths");
    GEOB_REQUIRE(net->num_stages >= 2 && net->num_stages <= GEOB200_MAX_STAGES, "backbone: num_stages out of range");
    GEOB_REQUIRE(n_pairs >= 1 && 2 * n_pairs <= GEOB_MAX_CLOUDS, "backbone: 1 <= pairs per batch <= %d", GEOB_MAX_CLOUDS / 2);
    GEOB_REQUIRE(n_pairs == 1 || cloud_rows_h != nullptr, "backbone: batched execution needs the per-cloud row counts of every level");
    Ctx c(workspace, workspace_bytes);
    c.gn_ws = gn_workspace; c.gn_ws_bytes = gn_workspace_bytes; c.stream = stream; c.groups = net->groups;
    const int S = net->num_stages;
    // per-level segmentation of the GroupNorm statistics: one segment per level for a single pair, else per pair
    GnSeg sg[GEOB200_MAX_STAGES];
    for (int l = 0; l < S; ++l) {
        GnSeg& g = sg[l];
        if (n_pairs == 1) {
            g = gn_one_segment(level_rows[l]);
            continue;
        }
        g.n_pairs = (int)n_pairs; g.n_clouds = (int)(2 * n_pairs); g.start[0] = 0;
        for (int cl = 0; cl < g.n_clouds; ++cl) g.start[cl + 1] = g.start[cl] + (int)cloud_rows_h[l][cl];
        GEOB_REQUIRE(g.start[g.n_clouds] == level_rows[l], "backbone: cloud rows of level %d do not add up", l);
    }
    const float* enc[GEOB200_MAX_STAGES];
    int64_t enc_ch[GEOB200_MAX_STAGES];
    // encoder1_1 (ConvBlock) + encoder1_2
    {
        const int64_t n0 = level_rows[0];
        float* yn = c.fl(n0, net->conv1.c_out);
        GEOB_REQUIRE(c.ar.ok(), "native: arena too small (encoder1_1)");
        TRY(run_kpconv_norm(c, net->conv1, net->norm1, feats, points[0], points[0], neighbors[0], n0, n0, neighbor_width[0], yn, sg[0]));
        const geob200_resblock_t& b = net->blocks[0];
        float* o = c.fl(n0, b.unary2.c_out);
        TRY(run_resblock(c, b, yn, n0, points[0], points[0], neighbors[0], n0, neighbor_width[0], o, sg[0], sg[0]));
        enc[0] = o; enc_ch[0] = b.unary2.c_out;
    }
    int bi = 1;
    for (int lvl = 1; lvl < S; ++lvl) {
        const int64_t m = level_rows[lvl], ns = level_rows[lvl - 1];
        const geob200_resblock_t& b1 = net->blocks[bi++];
        float* o1 = c.fl(m, b1.unary2.c_out);
        TRY(run_resblock(c, b1, enc[lvl - 1], ns, points[lvl], points[lvl - 1], subsampling[lvl - 1], m, subsampling_width[lvl - 1], o1,
                         sg[lvl - 1], sg[lvl], n_pairs > 1 ? sub_cloud_max[lvl - 1] : nullptr));
        const geob200_resblock_t& b2 = net->blocks[bi++];
        float* o2 = c.fl(m, b2.unary2.c_out);
        TRY(run_resblock(c, b2, o1, m, points[lvl], points[lvl], neighbors[lvl], m, neighbor_width[lvl], o2, sg[lvl], sg[lvl]));
        const geob200_resblock_t& b3 = net->blocks[bi++];
        float* o3 = (lvl == S - 1) ? out_feats[0] : c.fl(m, b3.unary2.c_out);
        TRY(run_resblock(c, b3, o2, m, points[lvl], points[lvl], neighbors[lvl], m, neighbor_width[lvl], o3, sg[lvl], sg[lvl]));
        enc[lvl] = o3; enc_ch[lvl] = b3.unary2.c_out;
    }
    // decoders: level S-1 (1-based) down to finest_decoder
    const float* latent = enc[S - 1];
    int64_t latent_ch = enc_ch[S - 1];
    int oi = 1;
    for (int lvl = S - 1; lvl >= net->finest_decoder; --lvl) {      // decoder{lvl}: output lives at level index lvl-1
        const int64_t m = level_rows[lvl - 1], ns = level_rows[lvl];
        const int64_t c2 = enc_ch[lvl - 1];
        float* cat = c.fl(m, latent_ch + c2);
        GEOB_REQUIRE(c.ar.ok(), "native: arena too small (decoder)");
        TRY(geob200_upsample_concat(latent, upsampling[lvl - 1], upsampling_width[lvl - 1], ns, enc[lvl - 1], m, latent_ch, c2, cat, stream));
        const geob200_linear_t& l = net->decoders[S - 1 - lvl];
        float* o = out_feats[oi++];
        if (lvl == net->finest_decoder) {
            TRY(geob200_linear(cat, l.c_in, l.weight, l.bias, o, l.c_out, m, l.c_out, l.c_in, 0, stream));
        } else {
            TRY(run_unary(c, l, net->decoder_norms[S - 1 - lvl], cat, m, nullptr, 1, o, sg[lvl - 1]));
        }
        latent = o; latent_ch = l.c_out;
    }
    GEOB_REQUIRE(c.ar.ok(), "native: arena too small");
    return 0;
}

// ---- transformer -------------------------------------------------------------------------------------------

size_t geob200_transformer_workspace_bytes(int64_t n0, int64_t n1, int64_t channels, int64_t heads, int64_t num_layers) {
    const int64_t rows[2] = {n0, n1};
    return geob200_transformer_batched_workspace_bytes(1, rows, channels, heads, num_layers);
}

static int run_tail(Ctx& c, const geob200_tlayer_t& L, const float* hidden, const float* inp, int64_t rows, int64_t ch, float* out) {
    float* h = c.fl(rows, ch);
    float* x = c.fl(rows, ch);
    float* y1 = c.fl(rows, 2 * ch);
    float* y2 = c.fl(rows, ch);
    GEOB_REQUIRE(c.ar.ok(), "native: arena too small (transformer tail)");
    TRY(geob200_linear(hidden, ch, L.att_linear.weight, L.att_linear.bias, h, ch, rows, ch, ch, 0, c.stream));
    TRY(geob200_add_layernorm(h, inp, L.att_norm.gamma, L.att_norm.beta, rows, ch, 1e-5f, x, c.stream));
    TRY(geob200_linear(x, ch, L.expand.weight, L.expand.bias, y1, 2 * ch, rows, 2 * ch, ch, 1, c.stream));
    TRY(geob200_linear(y1, 2 * ch, L.squeeze.weight, L.squeeze.bias, y2, ch, rows, ch, 2 * ch, 0, c.stream));
    TRY(geob200_add_layernorm(x, y2, L.out_norm.gamma, L.out_norm.beta, rows, ch, 1e-5f, out, c.stream));
    return 0;
}

// x: stacked [feats0; feats1] (n0+n1, C) hidden features (after in_proj); emb0 (n0,n0,C), emb1 (n1,n1,C); out (n0+n1, C).
int geob200_transformer_forward(const geob200_tlayer_t* layers, int64_t num_layers, int64_t channels, int64_t heads, const float* x_in,
                                int64_t n0, int64_t n1, const float* emb0, const float* emb1, float* out, void* workspace,
                                size_t workspace_bytes, void* stream) {
    const int64_t rows[2] = {n0, n1};
    const float* embs[2] = {emb0, emb1};
    return geob200_transformer_forward_batched(layers, num_layers, channels, heads, x_in, 1, rows, embs, out, workspace, workspace_bytes, stream);
}

size_t geob200_transformer_batched_workspace_bytes(int64_t n_pairs, const int64_t* cloud_rows_h, int64_t channels, int64_t heads,
                                                   int64_t num_layers) {
    size_t n = 0, att = 0;
    for (int64_t c = 0; c < 2 * n_pairs; ++c) {
        n += (size_t)cloud_rows_h[c];
        const size_t other = (size_t)cloud_rows_h[(c + n_pairs) % (2 * n_pairs)];
        const size_t m = (size_t)cloud_rows_h[c] > other ? (size_t)cloud_rows_h[c] : other;
        att += align_up((size_t)cloud_rows_h[c] * m * (size_t)heads * 4, 256);     // self (rows x rows) or cross (rows x partner rows)
    }
    return (n * (size_t)channels * 4 * (3 + 1 + (size_t)heads + 12)) * (size_t)(num_layers + 1) + att + (2 << 20);
}

// Batched form: x rows in stack order [ref_1..ref_B, src_1..src_B] (cloud_rows_h[2B]); embeddings[c] = structure embedding of
// cloud c (rows_c, rows_c, C).  Every Linear / LayerNorm runs ONCE over the rows of all pairs (the ref block and the src block
// are contiguous, so the cross-attention projections are single GEMMs too); attention runs as one batched launch pair per
// phase with one item per cloud (self) or per pair (cross).
int geob200_transformer_forward_batched(const geob200_tlayer_t* layers, int64_t num_layers, int64_t channels, int64_t heads,
                                        const float* x_in, int64_t n_pairs, const int64_t* cloud_rows_h, const float* const* embeddings,
                                        float* out, void* workspace, size_t workspace_bytes, void* stream) {
    GEOB_REQUIRE(n_pairs >= 1 && 2 * n_pairs <= GEOB_MAX_CLOUDS, "transformer: 1 <= pairs per batch <= %d", GEOB_MAX_CLOUDS / 2);
    Ctx c(workspace, workspace_bytes);
    c.stream = stream;
    const int64_t C = channels, H = heads, B = n_pairs, NC = 2 * n_pairs;
    int64_t off[GEOB_MAX_CLOUDS + 1];
    off[0] = 0;
    for (int64_t i = 0; i < NC; ++i) off[i + 1] = off[i] + cloud_rows_h[i];
    const int64_t n = off[NC], R = off[B];           // all rows; rows of the ref block
    const float* x = x_in;
    geob200_att_item_t items[GEOB_MAX_CLOUDS];
    // score scratch of the streaming attention, reused by every layer: sized for the larger of the self / cross batches
    size_t att_ws_bytes = 0;
    {
        for (int64_t i = 0; i < NC; ++i) { items[i].n_query = cloud_rows_h[i]; items[i].n_key = cloud_rows_h[i]; }
        att_ws_bytes = geob200_attention_batched_workspace_bytes(items, NC, H);
        for (int64_t p = 0; p < B; ++p) { items[p].n_query = cloud_rows_h[p]; items[p].n_key = cloud_rows_h[B + p]; }
        const size_t cross = geob200_attention_batched_workspace_bytes(items, B, H);
        if (cross > att_ws_bytes) att_ws_bytes = cross;
    }
    void* att_ws = c.fl((int64_t)(att_ws_bytes / 4 + 1), 1);
    for (int64_t i = 0; i < num_layers; ++i) {
        const geob200_tlayer_t& L = layers[i];
        float* y = (i == num_layers - 1) ? out : c.fl(n, C);
        if (L.is_self) {
            float* qkv = c.fl(n, 3 * C);
            float* qp = c.fl(n, H * C);
            float* qb = c.fl(n, H);
            float* hidden = c.fl(n, C);
            GEOB_REQUIRE(c.ar.ok(), "native: arena too small (self layer)");
            TRY(geob200_linear(x, C, L.w_qkv, L.b_qkv, qkv, 3 * C, n, 3 * C, C, 0, stream));
            const int64_t d = C / H;
            TRY(geob200_linear_batched(qkv, 3 * C, d, L.wp_t, C, d, nullptr, 0, qp, H * C, C, n, C, d, H, 0, stream));
            TRY(geob200_head_bias(qkv, 3 * C, L.bp, n, C, H, qb, stream));
            for (int64_t cl = 0; cl < NC; ++cl) {
                const int64_t o = off[cl];
                items[cl] = geob200_att_item_t{qkv + o * 3 * C, qkv + o * 3 * C + C, qkv + o * 3 * C + 2 * C, qp + o * H * C, qb + o * H,
                                               embeddings[cl], hidden + o * C, cloud_rows_h[cl], cloud_rows_h[cl]};
            }
            TRY(geob200_attention_batched(items, NC, 3 * C, 3 * C, 3 * C, C, C, H, att_ws, att_ws_bytes, stream));
            TRY(run_tail(c, L, hidden, x, n, C, y));
        } else {
            const int64_t Sn = n - R;
            float* q0 = c.fl(R, C);
            float* kv1 = c.fl(Sn, 2 * C);
            float* hid0 = c.fl(R, C);
            float* q1 = c.fl(Sn, C);
            float* kv0 = c.fl(R, 2 * C);
            float* hid1 = c.fl(Sn, C);
            GEOB_REQUIRE(c.ar.ok(), "native: arena too small (cross layer)");
            // feats0 <- layer(feats0, feats1) for every pair
            TRY(geob200_linear(x, C, L.w_q, L.b_q, q0, C, R, C, C, 0, stream));
            TRY(geob200_linear(x + R * C, C, L.w_kv, L.b_kv, kv1, 2 * C, Sn, 2 * C, C, 0, stream));
            for (int64_t p = 0; p < B; ++p) {
                const int64_t ro = off[p], so = off[B + p] - R;
                items[p] = geob200_att_item_t{q0 + ro * C, kv1 + so * 2 * C, kv1 + so * 2 * C + C, nullptr, nullptr, nullptr, hid0 + ro * C,
                                              cloud_rows_h[p], cloud_rows_h[B + p]};
            }
            TRY(geob200_attention_batched(items, B, C, 2 * C, 2 * C, C, C, H, att_ws, att_ws_bytes, stream));
            TRY(run_tail(c, L, hid0, x, R, C, y));
            // feats1 <- layer(feats1, UPDATED feats0)   (conditional_transformer.py:109-111, parallel=False)
            TRY(geob200_linear(x + R * C, C, L.w_q, L.b_q, q1, C, Sn, C, C, 0, stream));
            TRY(geob200_linear(y, C, L.w_kv, L.b_kv, kv0, 2 * C, R, 2 * C, C, 0, stream));
            for (int64_t p = 0; p < B; ++p) {
                const int64_t ro = off[p], so = off[B + p] - R;
                items[p] = geob200_att_item_t{q1 + so * C, kv0 + ro * 2 * C, kv0 + ro * 2 * C + C, nullptr, nullptr, nullptr, hid1 + so * C,
                                              cloud_rows_h[B + p], cloud_rows_h[p]};
            }
            TRY(geob200_attention_batched(items, B, C, 2 * C, 2 * C, C, C, H, att_ws, att_ws_bytes, stream));
            TRY(run_tail(c, L, hid1, x + R * C, Sn, C, y + R * C));
        }
        x = y;
    }
    return 0;
}

}  // extern "C"
