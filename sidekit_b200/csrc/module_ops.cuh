// Stand-alone module operators (SURVEY.md 8b "what a native replacement must export"): the same kernels the fused engine
// runs, behind entry points that take and return DENSE fp32 tensors, so that the reference's modules work on their own --
// BasicBlock / SELayer / ResBlock / PreHalfResNet34 (sidekit/nnet/res_net.py:186-320, :539-554), AttentivePooling
// (sidekit/nnet/pooling.py:151-171) and ArcMarginProduct(target=None) (sidekit/nnet/loss.py:299-310).
//
// Included at the end of engine.cu (it drives the engine's own geometry planner, conv launcher and plane exporter).
// A call converts its dense input into the engine's chunk-plane layout, runs the tcgen05 convolution (or the pooling
// kernels) and converts back; weights are folded / packed per call.  That makes these ops correct and native, not fast:
// the fast path is the fused engine, which never leaves the plane layout.
#pragma once

namespace skb {

// ----------------------------------------------------------------------------- dense NCHW fp32 -> chunk planes
// One thread per (pixel, 8-channel chunk).  Optional per-channel prologue x <- lrelu(x * s[c] + t[c], slope) (the
// pre-activation BatchNorm + LeakyReLU of ResBlock, res_net.py:238-241).  `pix_ps` != nullptr: the destination is the
// phase-split copy that feeds a stride-2 convolution (pixmeta tables, see planmeta_kernel).
template <bool BF16>
__global__ void pack_dense_kernel(const float* __restrict__ x, int B, int C, int H, int W, const float* __restrict__ pre_s,
                                  const float* __restrict__ pre_t, float pre_slope, uint16_t* __restrict__ dst, long long plane,
                                  int G, int Wp, const int* __restrict__ utt_row0, const int* __restrict__ pix_ps, int chunks,
                                  unsigned* __restrict__ overflow) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)B * H * W * chunks;
    if (idx >= total) return;
    const int w = (int)(idx % W);
    const int h = (int)((idx / W) % H);
    const int j = (int)((idx / ((long long)W * H)) % chunks);
    const int b = (int)(idx / ((long long)W * H * chunks));
    float v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        const int c = j * 8 + e;
        float t = 0.f;
        if (c < C) {
            t = x[(((size_t)b * C + c) * H + h) * W + w];
            if (pre_s != nullptr) {
                t = fmaf(t, pre_s[c], pre_t[c]);
                t = fmaxf(t, t * pre_slope);
            }
        }
        v[e] = t;
    }
    uint4 o;
    o.x = pack2<BF16>(v[0], v[1]); o.y = pack2<BF16>(v[2], v[3]); o.z = pack2<BF16>(v[4], v[5]); o.w = pack2<BF16>(v[6], v[7]);
    if (!BF16 && overflow != nullptr) {
        uint32_t m = 0u;
        track16(o, m);
        if (saturated16(m)) atomicAdd(overflow, 1u);
    }
    const int rel = (utt_row0[b] + h) * Wp + w;
    const long long pix = pix_ps != nullptr ? (long long)pix_ps[rel] : (long long)G + rel;
    *reinterpret_cast<uint4*>(dst + ((size_t)j * plane + pix) * 8) = o;
}

__global__ void fill_kernel(float* p, long long n, float v) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

// (B, C, H, W) -> (B, C) means: one CTA per (b, c), fixed-order block reduction (AdaptiveAvgPool2d(1), res_net.py:264, :279)
__global__ void __launch_bounds__(256) channel_mean_kernel(const float* __restrict__ x, long long hw, float* __restrict__ out) {
    __shared__ double red[8];
    const float* p = x + (size_t)blockIdx.x * hw;
    double s = 0.0;
    for (long long i = threadIdx.x; i < hw; i += blockDim.x) s += (double)p[i];
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < 8; ++i) t += red[i];
        out[blockIdx.x] = (float)(t / (double)hw);
    }
}

// scale[b][c] = sigmoid(W2 relu(W1 mean[b]))  (SELayer.fc, res_net.py:265-270); one CTA per batch item
__global__ void __launch_bounds__(256) se_gate_kernel(const float* __restrict__ mean, const float* __restrict__ fc1 /*[R][C]*/,
                                                      const float* __restrict__ fc2 /*[C][R]*/, int C, int R, float* __restrict__ scale) {
    extern __shared__ float sm[];              // [C] mean, [R] hidden
    float* hid = sm + C;
    const int b = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int c = threadIdx.x; c < C; c += blockDim.x) sm[c] = mean[(size_t)b * C + c];
    __syncthreads();
    for (int j = warp; j < R; j += blockDim.x >> 5) {
        float a = 0.f;
        for (int c = lane; c < C; c += 32) a = fmaf(fc1[(size_t)j * C + c], sm[c], a);
        a = warp_sum(a);
        if (lane == 0) hid[j] = fmaxf(a, 0.f);
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float a = 0.f;
        for (int j = 0; j < R; ++j) a = fmaf(fc2[(size_t)c * R + j], hid[j], a);
        scale[(size_t)b * C + c] = 1.f / (1.f + __expf(-a));
    }
}

// out = act(y * scale[b][c] + res): the tail of BasicBlock (res_net.py:316-319) / the whole of SELayer (scale only)
__global__ void scale_residual_act_kernel(const float* __restrict__ y, const float* __restrict__ scale, const float* __restrict__ res,
                                          long long hw, long long total, float slope, float* __restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    float v = y[i];
    if (scale != nullptr) v *= scale[i / hw];
    if (res != nullptr) v += res[i];
    out[i] = fmaxf(v, v * slope);
}

// x / max(||x||, eps) per row (torch.nn.functional.normalize, loss.py:304-305); one warp per row
__global__ void l2_normalize_kernel(const float* __restrict__ x, int N, int D, float eps, float* __restrict__ out) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= N) return;
    float s = 0.f;
    for (int k = lane; k < D; k += 32) s = fmaf(x[(size_t)row * D + k], x[(size_t)row * D + k], s);
    s = warp_sum(s);
    const float inv = 1.f / fmaxf(sqrtf(s), eps);
    for (int k = lane; k < D; k += 32) out[(size_t)row * D + k] = x[(size_t)row * D + k] * inv;
}

// (B, D, T) -> frame-major (B * T, D), tiled through shared memory
__global__ void bdt_to_frames_kernel(const float* __restrict__ x, int D, int T, float* __restrict__ X) {
    __shared__ float tile[32][33];
    const int b = blockIdx.z, d0 = blockIdx.y * 32, t0 = blockIdx.x * 32;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int d = d0 + i, t = t0 + threadIdx.x;
        tile[i][threadIdx.x] = (d < D && t < T) ? x[((size_t)b * D + d) * T + t] : 0.f;
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int t = t0 + i, d = d0 + threadIdx.x;
        if (t < T && d < D) X[((size_t)b * T + t) * D + d] = tile[threadIdx.x][i];
    }
}

// h = tanh(BN(relu(h + hb[frame / T]))) for a dense (B, T) frame grid (att_act_kernel with frame_utt = frame / T)
__global__ void att_act_dense_kernel(float* __restrict__ h, const float* __restrict__ hb, const float* __restrict__ bn_s,
                                     const float* __restrict__ bn_t, long long total, int A, int T) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int fr = (int)(idx / A), a = (int)(idx % A);
    const float x = h[idx] + hb[(size_t)(fr / T) * A + a];
    const float v = x > 0.f ? x : (x == x ? 0.f : x);       // NaN-transparent ReLU, as in att_act_kernel
    h[idx] = tanhf(fmaf(v, bn_s[a], bn_t[a]));
}

// softmax over time + weighted mean / std (pooling.py:167-169) on fp32 frames: one thread per (b, d), online softmax
__global__ void softmax_pool_dense_kernel(const float* __restrict__ X, const float* __restrict__ logit, int D, int T,
                                          float* __restrict__ out) {
    const int d = blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.y;
    if (d >= D) return;
    float m = -INFINITY, se = 0.f, sx = 0.f, sxx = 0.f;
    for (int t = 0; t < T; ++t) {
        const size_t o = ((size_t)b * T + t) * D + d;
        const float l = logit[o], x = X[o];
        if (l > m) {
            const float r = __expf(m - l);
            se *= r; sx *= r; sxx *= r;
            m = l;
        }
        const float e = __expf(l - m);
        se += e;
        sx = fmaf(x, e, sx);
        sxx = fmaf(x * x, e, sxx);
    }
    const float mu = sx / se;
    out[(size_t)b * 2 * D + d] = mu;
    out[(size_t)b * 2 * D + D + d] = sqrtf(fmaxf(sxx / se - mu * mu, 1e-9f));
}

// The per-(thread, device) scratch extractor handle the stand-alone convolution drives: no model, only a geometry plan,
// its tables and the overflow counter.
static skb_xtractor* ops_context() {
    static thread_local skb_xtractor* ctx[kMaxDevices] = {};
    const int d = current_device();
    if (!ctx[d]) {
        skb_xtractor* h = new skb_xtractor();
        h->device = d;
        h->m.archi = SKB_ARCHI_HALFRESNET34;
        if (h->ovf.ensure(sizeof(unsigned)) != SKB_OK || cudaMemset(h->ovf.p, 0, sizeof(unsigned)) != cudaSuccess) {
            delete h;
            return nullptr;
        }
        ctx[d] = h;
    }
    return ctx[d];
}

static int conv_cout_pad(int cout) { return cout <= 32 ? 32 : (cout <= 64 ? 64 : (cout + 127) / 128 * 128); }

}  // namespace skb

extern "C" {

int skb_conv2d_bn_act(const float* x_dev, int B, int Cin, int H, int W, const float* w_host, const float* bias_host, int Cout,
                      int ksize, int stride, const float* pre_scale_dev, const float* pre_shift_dev, float pre_slope,
                      float act_slope, const float* se_scale_dev, const float* residual_dev, int compute_dtype, float* y_dev,
                      void* stream) {
    if (!x_dev || !w_host || !bias_host || !y_dev || B <= 0 || Cin <= 0 || Cout <= 0 || H <= 0 || W <= 0 ||
        (ksize != 1 && ksize != 3) || (stride != 1 && stride != 2) || act_slope < 0.f || act_slope > 1.f) {
        set_last_error(__FILE__, __LINE__, "conv2d_bn_act: bad arguments (3x3 pad 1 or 1x1 pad 0, stride 1 or 2, 0 <= slope <= 1)");
        return SKB_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    skb_xtractor* h = ops_context();
    if (!h) {
        set_last_error(__FILE__, __LINE__, "conv2d_bn_act: cannot create the operator context");
        return SKB_ERR_CUDA;
    }
    const bool bf16 = compute_dtype == 1;
    h->m.bf16 = bf16;
    const int taps = ksize * ksize;
    const int cin_pad = (Cin + kConvKC - 1) / kConvKC * kConvKC, cout_pad = conv_cout_pad(Cout);
    const int Ho = stride == 2 ? (H - 1) / 2 + 1 : H, Wo = stride == 2 ? (W - 1) / 2 + 1 : W;
    // ---- geometry: the input level, and for stride 2 the output level whose phase-split copy the convolution reads
    Plan& pl = h->plan;
    pl = Plan();
    pl.B = B;
    pl.lv.resize(stride == 2 ? 2 : 1);
    h->m.level_halves[0] = false;
    h->m.level_halves[1] = stride == 2;
    plan_level(&pl, &pl.lv[0], W, cin_pad, std::vector<int>((size_t)B, H), true, W + 2);
    if (stride == 2) plan_level(&pl, &pl.lv[1], Wo, cout_pad, std::vector<int>((size_t)B, Ho), true, Wo + 2);
    SKB_TRY(h->slot.tab32.ensure(pl.tab32.size() * sizeof(int)));
    SKB_CUDA_CHECK(cudaMemcpyAsync(h->slot.tab32.p, pl.tab32.data(), pl.tab32.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    SKB_CUDA_CHECK(cudaStreamSynchronize(st));                // pl.tab32 is pageable
    h->d32 = (const int*)h->slot.tab32.p;
    SKB_TRY(build_pixmeta(h, st));
    const Level& L0 = pl.lv[0];
    const Level& Lg = pl.lv[stride == 2 ? 1 : 0];              // the geometry the convolution walks = its output geometry
    const int* pm = (const int*)h->slot.pixmeta.p;
    // ---- buffers: input planes (or phase-split input), output planes, residual planes, padded SE scale table
    h->act.resize(3);
    const size_t in_bytes = stride == 2 ? (size_t)4 * (cin_pad / 8) * Lg.plane * 16 : (size_t)(cin_pad / 8) * L0.plane * 16;
    const size_t out_bytes = (size_t)(cout_pad / 8) * Lg.plane * 16;
    SKB_TRY(h->act[0].ensure(in_bytes));
    SKB_TRY(h->act[1].ensure(out_bytes));
    SKB_TRY(h->act[2].ensure(out_bytes));
    SKB_CUDA_CHECK(cudaMemsetAsync(h->act[0].p, 0, in_bytes, st));
    const bool fused = se_scale_dev != nullptr || residual_dev != nullptr;
    if (fused) SKB_CUDA_CHECK(cudaMemsetAsync(h->act[2].p, 0, out_bytes, st));
    {
        const long long total = (long long)B * H * W * (cin_pad / 8);
        const unsigned blocks = (unsigned)((total + 255) / 256);
        const int* ps = stride == 2 ? pm + L0.o_pix_sub : nullptr;
        const long long plane = stride == 2 ? Lg.plane : L0.plane;
        SKB_CUDA_CHECK(launch_kernel(false, bf16 ? pack_dense_kernel<true> : pack_dense_kernel<false>, blocks, 256, 0, st, x_dev, B, Cin, H, W,
                                     pre_scale_dev, pre_shift_dev, pre_slope, (uint16_t*)h->act[0].p, plane, L0.G, L0.Wp,
                                     h->d32 + L0.o_utt_row0, ps, cin_pad / 8, (unsigned*)h->ovf.p));
    }
    const float* scale = nullptr;
    if (fused) {
        if (residual_dev != nullptr) {
            const long long total = (long long)B * Ho * Wo * (cout_pad / 8);
            const unsigned blocks = (unsigned)((total + 255) / 256);
            SKB_CUDA_CHECK(launch_kernel(false, bf16 ? pack_dense_kernel<true> : pack_dense_kernel<false>, blocks, 256, 0, st, residual_dev, B,
                                         Cout, Ho, Wo, nullptr, nullptr, 1.f, (uint16_t*)h->act[2].p, Lg.plane, Lg.G, Lg.Wp,
                                         h->d32 + Lg.o_utt_row0, nullptr, cout_pad / 8, nullptr));
        }
        SKB_TRY(h->scale.ensure((size_t)B * cout_pad * sizeof(float)));
        const long long n = (long long)B * cout_pad;
        SKB_CUDA_CHECK(launch_kernel(false, fill_kernel, (unsigned)((n + 255) / 256), 256, 0, st, (float*)h->scale.p, n, 1.f));
        if (se_scale_dev != nullptr)
            SKB_CUDA_CHECK(cudaMemcpy2DAsync(h->scale.p, (size_t)cout_pad * sizeof(float), se_scale_dev, (size_t)Cout * sizeof(float),
                                             (size_t)Cout * sizeof(float), B, cudaMemcpyDeviceToDevice, st));
        scale = (const float*)h->scale.p;
    }
    // ---- weights: zero-padded to (cout_pad, cin_pad), packed for the tcgen05 kernel
    std::vector<double> wf((size_t)cout_pad * cin_pad * taps, 0.0), bias((size_t)cout_pad, 0.0);
    for (int co = 0; co < Cout; ++co) {
        bias[co] = bias_host[co];
        for (int ci = 0; ci < Cin; ++ci)
            for (int t = 0; t < taps; ++t) wf[((size_t)co * cin_pad + ci) * taps + t] = w_host[((size_t)co * Cin + ci) * taps + t];
    }
    ConvW cw;
    int rc;
    int kind;
    if (stride == 2 && ksize == 3) {
        rc = pack_conv_phase_split(wf, bias, cout_pad, cin_pad, bf16, &cw);
        kind = 3;
    } else {
        rc = pack_conv(wf, bias, cout_pad, cin_pad, cin_pad, taps, bf16, &cw);
        kind = ksize == 3 ? 1 : 0;
    }
    if (rc) { free_conv(&cw); return rc; }
    h->slope_override = act_slope;
    rc = run_conv(h, cw, kind, Lg, (const uint16_t*)h->act[0].p, (uint16_t*)h->act[1].p, 0, nullptr, scale,
                  fused ? (const uint16_t*)h->act[2].p : nullptr, nullptr, nullptr, st);
    h->slope_override = -1.f;
    if (!rc) {
        Level Lx = Lg;
        Lx.C = Cout;                                           // export the real channels only
        int64_t per = 0;
        rc = export_stage(h, (const uint16_t*)h->act[1].p, Lx, Ho, y_dev, &per, st);
    }
    // a failed launch in run_conv / export_stage has recorded its own file:line; the packed weights are freed below
    if (!rc) {
        const cudaError_t e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) { set_last_error(__FILE__, __LINE__, cudaGetErrorString(e)); rc = SKB_ERR_CUDA; }
    }
    free_conv(&cw);
    return rc;
}

int skb_ops_overflow_count(void* stream, int64_t* count) {
    skb_xtractor* h = ops_context();
    if (!h || !count) {
        set_last_error(__FILE__, __LINE__, "ops_overflow_count: bad arguments");
        return SKB_ERR_ARG;
    }
    return skb_xtractor_overflow_count(h, stream, count);
}

int skb_channel_mean(const float* x_dev, int B, int C, int64_t hw, float* out_dev, void* stream) {
    if (!x_dev || !out_dev || B <= 0 || C <= 0 || hw <= 0) {
        set_last_error(__FILE__, __LINE__, "channel_mean: bad arguments");
        return SKB_ERR_ARG;
    }
    SKB_CUDA_CHECK(launch_kernel(false, channel_mean_kernel, B * C, 256, 0, (cudaStream_t)stream, x_dev, (long long)hw, out_dev));
    return SKB_OK;
}

int skb_se_gate(const float* mean_dev, const float* fc1_dev, const float* fc2_dev, int B, int C, int R, float* scale_dev, void* stream) {
    if (!mean_dev || !fc1_dev || !fc2_dev || !scale_dev || B <= 0 || C <= 0 || R <= 0) {
        set_last_error(__FILE__, __LINE__, "se_gate: bad arguments");
        return SKB_ERR_ARG;
    }
    SKB_CUDA_CHECK(launch_kernel(false, se_gate_kernel, B, 256, (size_t)(C + R) * sizeof(float), (cudaStream_t)stream, mean_dev, fc1_dev,
                                 fc2_dev, C, R, scale_dev));
    return SKB_OK;
}

int skb_scale_residual_act(const float* y_dev, const float* scale_dev, const float* res_dev, int B, int C, int64_t hw, float slope,
                           float* out_dev, void* stream) {
    if (!y_dev || !out_dev || B <= 0 || C <= 0 || hw <= 0) {
        set_last_error(__FILE__, __LINE__, "scale_residual_act: bad arguments");
        return SKB_ERR_ARG;
    }
    const long long total = (long long)B * C * hw;
    SKB_CUDA_CHECK(launch_kernel(false, scale_residual_act_kernel, (unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream, y_dev,
                                 scale_dev, res_dev, (long long)hw, total, slope, out_dev));
    return SKB_OK;
}

int skb_l2_normalize(const float* x_dev, int N, int D, float eps, float* out_dev, void* stream) {
    if (!x_dev || !out_dev || N <= 0 || D <= 0) {
        set_last_error(__FILE__, __LINE__, "l2_normalize: bad arguments");
        return SKB_ERR_ARG;
    }
    SKB_CUDA_CHECK(launch_kernel(false, l2_normalize_kernel, (N + 7) / 8, 256, 0, (cudaStream_t)stream, x_dev, N, D, eps, out_dev));
    return SKB_OK;
}

int skb_attentive_pool(const float* x_dev, int B, int D, int T, const float* w1_dev, const float* b1_dev, const float* bn_s_dev,
                       const float* bn_t_dev, const float* w2_dev, const float* b2_dev, int A, int global_context, float* out_dev,
                       void* stream) {
    if (!x_dev || !w1_dev || !b1_dev || !bn_s_dev || !bn_t_dev || !w2_dev || !b2_dev || !out_dev || B <= 0 || D <= 0 || T <= 0 || A <= 0) {
        set_last_error(__FILE__, __LINE__, "attentive_pool: bad arguments");
        return SKB_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int in_factor = global_context ? 3 : 1;
    const size_t F = (size_t)B * T;
    DevBuf X, Hh, Lg, gc, hb, w1x, w1g, ws;
    auto release = [&]() { X.release(); Hh.release(); Lg.release(); gc.release(); hb.release(); w1x.release(); w1g.release(); ws.release(); };
    int rc = SKB_OK;
    PackedOp p1, p2;
    do {
        if ((rc = X.ensure(F * D * sizeof(float))) || (rc = Hh.ensure(F * A * sizeof(float))) || (rc = Lg.ensure(F * D * sizeof(float))) ||
            (rc = hb.ensure((size_t)B * A * sizeof(float))) || (rc = w1x.ensure((size_t)A * D * sizeof(float)))) break;
        if (launch_kernel(false, bdt_to_frames_kernel, dim3((T + 31) / 32, (D + 31) / 32, B), dim3(32, 8), 0, st, x_dev, D, T, (float*)X.p) !=
            cudaSuccess) { rc = SKB_ERR_CUDA; break; }
        // split the first Conv1d's weight (A, in_factor * D) into the part that multiplies x and the time-constant part
        if (cudaMemcpy2DAsync(w1x.p, (size_t)D * sizeof(float), w1_dev, (size_t)in_factor * D * sizeof(float), (size_t)D * sizeof(float), A,
                              cudaMemcpyDeviceToDevice, st) != cudaSuccess) { rc = SKB_ERR_CUDA; break; }
        if (global_context) {
            if ((rc = gc.ensure((size_t)B * 2 * D * sizeof(float))) || (rc = w1g.ensure((size_t)A * 2 * D * sizeof(float)))) break;
            if (cudaMemcpy2DAsync(w1g.p, (size_t)2 * D * sizeof(float), w1_dev + D, (size_t)3 * D * sizeof(float), (size_t)2 * D * sizeof(float),
                                  A, cudaMemcpyDeviceToDevice, st) != cudaSuccess) { rc = SKB_ERR_CUDA; break; }
            if ((rc = skb_meanstd_pool(x_dev, B, D, T, (float*)gc.p, stream))) break;       // [mean ; unbiased std] over time
            if ((rc = ws.ensure(skinny_gemm_ws_floats(B, A, 2 * D) * sizeof(float)))) break;
            if ((rc = launch_skinny_gemm((const float*)gc.p, B, 2 * D, (const float*)w1g.p, A, b1_dev, 1.f, (float*)hb.p, A, (float*)ws.p, st))) break;
        } else if ((rc = launch_broadcast_rows(b1_dev, B, A, (float*)hb.p, st))) break;
        if ((rc = packed_create((const float*)w1x.p, A, D, &p1, st))) break;
        if ((rc = packed_create(w2_dev, D, A, &p2, st))) break;
        if ((rc = gemm_nt_split((const float*)X.p, (int)F, D, p1, nullptr, 1.f, (float*)Hh.p, A, st))) break;
        const long long total = (long long)F * A;
        if (launch_kernel(false, att_act_dense_kernel, (unsigned)((total + 255) / 256), 256, 0, st, (float*)Hh.p, (const float*)hb.p, bn_s_dev,
                          bn_t_dev, total, A, T) != cudaSuccess) { rc = SKB_ERR_CUDA; break; }
        if ((rc = gemm_nt_split((const float*)Hh.p, (int)F, A, p2, b2_dev, 1.f, (float*)Lg.p, D, st))) break;
        if (launch_kernel(false, softmax_pool_dense_kernel, dim3((D + 127) / 128, B), 128, 0, st, (const float*)X.p, (const float*)Lg.p, D, T,
                          out_dev) != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess) rc = SKB_ERR_CUDA;
    } while (false);
    if (rc == SKB_ERR_CUDA) set_last_error(__FILE__, __LINE__, cudaGetErrorString(cudaGetLastError()));
    cudaStreamSynchronize(st);
    packed_free(&p1);
    packed_free(&p2);
    release();
    return rc;
}

}  // extern "C"
