// Load-time weight folding and packing (host side). Replaces the reference's texture repacks
// Conv2DLayer::oihw2hwo4i4 (core/src/ic2/conv2d.cpp:76-100) and SeparableConv2DLayer::oihw2hwo4i4
// (separableconvolution.cpp:88-111), and moves BatchNorm out of the shader epilogue
// (shadertemplate_vk_conv2d.comp:277-288) into the weights:
//     s = max(sqrt(var + 1e-3), 1e-4);  scale = gamma / s;
//     y = scale*(conv + bias - mean) + beta  =  conv(w*scale) + ((bias - mean)*scale + beta)
#include <cmath>
#include <cstring>

#include "snnb_internal.h"

namespace snnb {

static inline size_t align256(size_t v) { return (v + 255) & ~(size_t) 255; }

size_t PackedHost::device_bytes() const {
    size_t b = 0;
    b += align256(w_f32.size() * sizeof(float));
    b += align256(w_hi.size() * sizeof(__half));
    b += align256(w_lo.size() * sizeof(__half));
    b += align256(w_row_hi.size() * sizeof(__half));
    b += align256(w_row_lo.size() * sizeof(__half));
    b += align256(w_feed_hi.size() * sizeof(__half));
    b += align256(w_feed_lo.size() * sizeof(__half));
    b += align256(bias.size() * sizeof(float));
    b += align256(gamma.size() * sizeof(float));
    b += align256(beta.size() * sizeof(float));
    b += align256(mean.size() * sizeof(float));
    b += align256(var.size() * sizeof(float));
    return b;
}

static void bn_fold(int OC, const float* bias, const float* g, const float* b, const float* m, const float* v, std::vector<float>& scale,
                    std::vector<float>& shift) {
    scale.assign(OC, 1.0f);
    shift.assign(OC, 0.0f);
    const bool has_bn = (m != nullptr) || (v != nullptr) || (g != nullptr) || (b != nullptr);
    for (int o = 0; o < OC; ++o) {
        const float bi = bias ? bias[o] : 0.0f;
        if (has_bn) {
            const float gamma = g ? g[o] : 1.0f, beta = b ? b[o] : 0.0f, mean = m ? m[o] : 0.0f, var = v ? v[o] : 1.0f;
            float s  = std::sqrt(var + 0.001f);
            s        = std::max(s, 0.0001f);
            scale[o] = gamma / s;
            shift[o] = (bi - mean) * scale[o] + beta;
        } else {
            shift[o] = bi;
        }
    }
}

void pack_conv2d_host(int IC, int OC, int k, const float* w_oihw, const float* bias, const float* g, const float* b, const float* m, const float* v,
                      PackedHost& out) {
    out.kind = 1, out.in_ch = IC, out.out_ch = OC, out.kernel = k;
    std::vector<float> scale, shift;
    bn_fold(OC, bias, g, b, m, v, scale, shift);
    const int K = k * k * IC;
    // tcgen05 operand: row = oc, column = tap*ICp + ic with ICp = round_up(IC, 8), so that every tap starts on a
    // 16-byte boundary (TMA box start) and the padding columns are zero.
    const int ICp = round_up(IC, 8);
    out.ocw     = round_up(OC, 64);
    out.kp      = k * k * ICp;
    out.ocr     = round_up(OC, 16);
    out.w_f32.assign((size_t) K * out.ocw, 0.0f);
    out.w_hi.assign((size_t) out.ocr * out.kp, __float2half_rn(0.0f));
    out.w_lo.assign((size_t) out.ocr * out.kp, __float2half_rn(0.0f));
    out.bias.assign(out.ocw + 320, 0.0f); // zero tail: the tcgen05 epilogue reads float4s up to tiles_oc * n_blk (n_blk <= 256)
    for (int o = 0; o < OC; ++o) {
        out.bias[o] = shift[o];
        for (int i = 0; i < IC; ++i)
            for (int ky = 0; ky < k; ++ky)
                for (int kx = 0; kx < k; ++kx) {
                    const float wv  = w_oihw[(((size_t) o * IC + i) * k + ky) * k + kx] * scale[o];
                    const int kidx  = (ky * k + kx) * IC + i;
                    out.w_f32[(size_t) kidx * out.ocw + o] = wv;
                    const int kcol                         = (ky * k + kx) * ICp + i;
                    const __half h                  = __float2half_rn(wv);
                    out.w_hi[(size_t) o * out.kp + kcol]   = h;
                    out.w_lo[(size_t) o * out.kp + kcol]   = __float2half_rn(wv - __half2float(h));
                }
    }
}

void pack_shortcut_host(int IC, const float* w_oi, const float* bias, const float* g, const float* b, const float* m, const float* v, PackedHost& out) {
    const int OC = out.out_ch;
    std::vector<float> scale, shift;
    bn_fold(OC, bias, g, b, m, v, scale, shift);
    // [OCr][kp] -> [OCr][kp + ICp]: the shortcut's columns follow the taps', in the order the producer walks its K blocks
    const int kp = out.kp + round_up(IC, 8);
    std::vector<__half> hi((size_t) out.ocr * kp, __float2half_rn(0.0f)), lo((size_t) out.ocr * kp, __float2half_rn(0.0f));
    for (int o = 0; o < out.ocr; ++o) {
        std::memcpy(&hi[(size_t) o * kp], &out.w_hi[(size_t) o * out.kp], out.kp * sizeof(__half));
        std::memcpy(&lo[(size_t) o * kp], &out.w_lo[(size_t) o * out.kp], out.kp * sizeof(__half));
    }
    for (int o = 0; o < OC; ++o) {
        out.bias[o] += shift[o];
        for (int i = 0; i < IC; ++i) {
            const float wv  = w_oi[(size_t) o * IC + i] * scale[o];
            const __half h  = __float2half_rn(wv);
            const size_t at = (size_t) o * kp + out.kp + i;
            hi[at] = h;
            lo[at] = __float2half_rn(wv - __half2float(h));
        }
    }
    out.w_hi.swap(hi), out.w_lo.swap(lo);
    out.kp = kp;
}

void pack_rowwin_host(PackedHost& p, int stride, int pad_x) {
    RowPlan rp;
    if (p.kind != 1 || p.in_ch > 8 || p.out_ch > 64 || !make_row_plan(p.kernel, stride, pad_x, rp)) return;
    const int k = p.kernel, IC = p.in_ch, OC = p.out_ch;
    p.row_stride = stride, p.row_pad = pad_x;
    const int panels = (rp.ksteps + 3) / 4; // 64 K columns (4 K steps) per panel: [ky][panel][OCr][64]
    p.w_row_hi.assign((size_t) k * panels * p.ocr * 64, __float2half_rn(0.0f));
    p.w_row_lo.assign((size_t) k * panels * p.ocr * 64, __float2half_rn(0.0f));
    for (int ky = 0; ky < k; ++ky)
        for (int o = 0; o < OC; ++o)
            for (int q = 0; q < rp.ksteps; ++q)
                for (int h = 0; h < 2; ++h) {
                    const int j = rp.ks_tap[q][h];
                    if (j < 0) continue;
                    for (int c = 0; c < IC; ++c) {
                        const float wv        = p.w_f32[(size_t) ((ky * k + j) * IC + c) * p.ocw + o]; // BN already folded in
                        const size_t idx      = (((size_t) ky * panels + q / 4) * p.ocr + o) * 64 + (q % 4) * 16 + h * 8 + c;
                        const __half hh = __float2half_rn(wv);
                        p.w_row_hi[idx]       = hh;
                        p.w_row_lo[idx]       = __float2half_rn(wv - __half2float(hh));
                    }
                }
}

void pack_feed_host(PackedHost& p, int stride, int pad_x) {
    FeedPlan fp;
    if (p.kind != 1 || p.out_ch > 64 || p.w_row_hi.empty() || !make_feed_plan(p.kernel, stride, pad_x, p.in_ch, fp)) return;
    const int k = p.kernel, IC = p.in_ch, OC = p.out_ch;
    p.feed_pad = pad_x;
    const int rpp = fp.rows_per_panel, prows = (k + rpp - 1) / rpp, sub = 64 / rpp; // filter rows per 128-byte weight row, K columns each
    p.w_feed_hi.assign((size_t) prows * p.ocr * 64, __float2half_rn(0.0f));
    p.w_feed_lo.assign((size_t) prows * p.ocr * 64, __float2half_rn(0.0f));
    for (int ky = 0; ky < k; ++ky)
        for (int o = 0; o < OC; ++o)
            for (int off = 0; off < 2 * fp.nch; ++off) { // pixel offset within the window = chunk off / 2, pixel off % 2
                const int t = off - fp.d;
                if (t < 0 || t >= k) continue;
                for (int c = 0; c < IC; ++c) {
                    const float wv   = p.w_f32[(size_t) ((ky * k + t) * IC + c) * p.ocw + o]; // BN already folded in
                    const size_t idx = ((size_t) (ky / rpp) * p.ocr + o) * 64 + (ky % rpp) * sub + off * 4 + c;
                    const __half hh  = __float2half_rn(wv);
                    p.w_feed_hi[idx] = hh;
                    p.w_feed_lo[idx] = __float2half_rn(wv - __half2float(hh));
                }
            }
}

void pack_depthwise_host(int C, int k, const float* w_chw, const float* bias, const float* g, const float* b, const float* m, const float* v,
                         PackedHost& out) {
    out.kind = 2, out.in_ch = C, out.out_ch = C, out.kernel = k;
    std::vector<float> scale, shift;
    bn_fold(C, bias, g, b, m, v, scale, shift);
    const int Cp = round_up(C, 8);
    out.ocw      = Cp;
    out.w_f32.assign((size_t) k * k * Cp, 0.0f);
    out.bias.assign(round_up(C, 64), 0.0f);
    for (int c = 0; c < C; ++c) {
        out.bias[c] = shift[c];
        for (int t = 0; t < k * k; ++t) out.w_f32[(size_t) t * Cp + c] = w_chw[(size_t) c * k * k + t] * scale[c];
    }
}

void pack_channels_host(int C, const float* g, const float* b, const float* m, const float* v, PackedHost& out) {
    out.kind = 4, out.in_ch = C, out.out_ch = C;
    const int Cp = round_up(C, 8);
    out.gamma.assign(Cp, 0.0f), out.beta.assign(Cp, 0.0f), out.mean.assign(Cp, 0.0f), out.var.assign(Cp, 0.0f);
    for (int c = 0; c < C; ++c) {
        out.gamma[c] = g ? g[c] : 1.0f;
        out.beta[c]  = b ? b[c] : 0.0f;
        out.mean[c]  = m ? m[c] : 0.0f;
        // the device never needs var itself: the `var` slot carries the BatchNormalization scale in the shader's
        // form, gamma / max(sqrt(var + 1e-3), 1e-4) (vk_batchnorm.comp:60-66); InstanceNorm reads the raw gamma/beta.
        float s      = std::sqrt((v ? v[c] : 1.0f) + 0.001f);
        s            = std::max(s, 0.0001f);
        out.var[c]   = out.gamma[c] / s;
    }
}

template <class T> static int put(snnb_context* ctx, const std::vector<T>& src, char*& cur, T** dst) {
    *dst = nullptr;
    if (src.empty()) return 0;
    *dst = reinterpret_cast<T*>(cur);
    SNNB_CUDA_OK(cudaMemcpyAsync(cur, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
    cur += align256(src.size() * sizeof(T));
    return 0;
}

int place_weights(snnb_context* ctx, const PackedHost& p, char* base, snnb_weights* w) {
    char* cur = base;
    w->ctx = ctx, w->kind = p.kind, w->in_ch = p.in_ch, w->out_ch = p.out_ch, w->kernel = p.kernel;
    w->ocw = p.ocw, w->kp = p.kp, w->ocr = p.ocr;
    w->row_stride = p.row_stride, w->row_pad = p.row_pad;
    if (put(ctx, p.w_f32, cur, &w->w_f32)) return 1;
    if (put(ctx, p.w_hi, cur, &w->w_hi)) return 1;
    if (put(ctx, p.w_lo, cur, &w->w_lo)) return 1;
    if (put(ctx, p.w_row_hi, cur, &w->w_row_hi)) return 1;
    if (put(ctx, p.w_row_lo, cur, &w->w_row_lo)) return 1;
    w->feed_pad = p.feed_pad;
    if (put(ctx, p.w_feed_hi, cur, &w->w_feed_hi)) return 1;
    if (put(ctx, p.w_feed_lo, cur, &w->w_feed_lo)) return 1;
    if (put(ctx, p.bias, cur, &w->bias)) return 1;
    if (put(ctx, p.gamma, cur, &w->gamma)) return 1;
    if (put(ctx, p.beta, cur, &w->beta)) return 1;
    if (put(ctx, p.mean, cur, &w->mean)) return 1;
    if (put(ctx, p.var, cur, &w->var)) return 1;
    // the source vectors live on the caller's stack/heap: make the async copies safe
    SNNB_CUDA_OK(cudaStreamSynchronize(ctx->stream));
    w->bytes = (size_t) (cur - base);
    return 0;
}

} // namespace snnb
