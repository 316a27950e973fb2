// Context, error reporting, Gaussian constants, the staging layouts and their weight pack kernels.
#include <math.h>
#include <stdarg.h>

#include "tg_umma.cuh"

static thread_local char g_err[512] = "";

void tg_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" const char *tg_last_error(void) { return g_err; }
extern "C" int tg_abi_version(void) { return TG_ABI_VERSION; }

extern "C" int tg_ctx_create(int device, tg_ctx **out) {
    TG_REQUIRE(out != nullptr, TG_ERR_ARG, "tg_ctx_create: out is null");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        tg_set_error("no CUDA device available (%s); this engine has no CPU fallback",
                     e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
        return TG_ERR_NO_DEVICE;
    }
    TG_REQUIRE(device >= 0 && device < count, TG_ERR_ARG, "device %d out of range [0,%d)", device, count);
    cudaDeviceProp prop;
    TG_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        tg_set_error("device %d is sm_%d%d; kernels are built for sm_100a only", device, prop.major, prop.minor);
        return TG_ERR_NO_DEVICE;
    }
    tg_ctx *c = new tg_ctx();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    c->smem_optin = (int)prop.sharedMemPerBlockOptin;
    c->packed = nullptr;
    c->packed_cap = 0;
    c->packed_tc = nullptr;
    c->packed_tc_cap = 0;
    c->math_mode = TG_MATH_AUTO;
    c->scratch = nullptr;
    c->scratch_cap = 0;
    c->order_buf = nullptr;
    c->order_cap = 0;
    c->perm = c->cnt = nullptr;
    *out = c;
    return TG_OK;
}

extern "C" void tg_ctx_destroy(tg_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->packed) cudaFree(ctx->packed);
    if (ctx->packed_tc) cudaFree(ctx->packed_tc);
    if (ctx->order_buf) cudaFree(ctx->order_buf);
    if (ctx->scratch) cudaFree(ctx->scratch);
    delete ctx;
}

extern "C" int tg_ctx_set_math(tg_ctx *ctx, int math_mode) {
    TG_REQUIRE(ctx != nullptr, TG_ERR_ARG, "tg_ctx_set_math: ctx is null");
    TG_REQUIRE(math_mode >= TG_MATH_AUTO && math_mode <= TG_MATH_3XTF32, TG_ERR_ARG, "unknown math mode %d", math_mode);
    ctx->math_mode = math_mode;
    return TG_OK;
}

// ---------------------------------------------------------------------------
// tensor-core staging
// ---------------------------------------------------------------------------
bool tg_tc_eligible(const tg_mlp_cfg *mlp) {
    if (!mlp || mlp->n_layers < 3 || mlp->n_layers > TG_MAX_LAYERS) return false;   // >= 2 hidden layers
    const int W = mlp->dims[1];
    if (W != 64 && W != 128) return false;
    for (int l = 1; l < mlp->n_layers; ++l)
        if (mlp->dims[l] != W) return false;
    // every hidden->hidden weight (hi + lo) is resident in shared memory next to the first/last layer rows
    if ((size_t)(mlp->n_layers - 2) * 2 * W * W * 4 > (size_t)160 * 1024) return false;
    return mlp->dims[0] >= 1 && mlp->dims[0] <= TG_MAX_OBS && mlp->dims[mlp->n_layers] >= 1 &&
           mlp->dims[mlp->n_layers] <= TG_MAX_ACT && mlp->activation >= 0 && mlp->activation <= 2;
}

int tg_build_tc_layout(const tg_mlp_cfg *mlp, tg_tc_layout *out, bool with_backward) {
    TG_REQUIRE(tg_tc_eligible(mlp), TG_ERR_UNSUPPORTED,
               "tensor-core path needs >= 2 hidden layers of equal width 64 or 128 whose weights fit in shared memory");
    memset(out, 0, sizeof(*out));
    const int nl = mlp->n_layers;
    out->n_layers = nl;
    out->W = mlp->dims[1];
    const int TCW = out->W;
    out->nh = nl - 1;
    out->act = mlp->activation;
    out->O = mlp->dims[0];
    out->O4 = tg_round_up(out->O + 1, 4);
    out->A = mlp->dims[nl];
    int64_t flat = 0;
    for (int l = 0; l < nl; ++l) {
        out->flat_w[l] = flat;
        flat += (int64_t)mlp->dims[l] * mlp->dims[l + 1] + mlp->dims[l + 1];
    }
    out->n_params = flat;
    int64_t off = 0;   // floats; MMA operand blocks 1024-byte (256-float) aligned
    for (int l = 1; l < nl - 1; ++l) {
        out->whi[l] = off; off += TCW * TCW;
        out->wlo[l] = off; off += TCW * TCW;
        out->wbhi[l] = out->wblo[l] = -1;
        if (with_backward) {
            out->wbhi[l] = off; off += TCW * TCW;
            out->wblo[l] = off; off += TCW * TCW;
        }
    }
    for (int l = 1; l < nl - 1; ++l) { out->bias[l] = off; off += TCW; }
    out->w1 = off; off += (int64_t)TCW * out->O4;
    out->wo = off; off += (int64_t)out->A * TCW;
    out->bo = off; off += 4;
    out->total = tg_round_up((int)off, 4);
    return TG_OK;
}

__global__ void pack_tc_kernel(tg_tc_layout lay, const float *__restrict__ params, float *__restrict__ packed) {
    const int nl = lay.n_layers, TCW = lay.W;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < lay.total;
         i += (int64_t)gridDim.x * blockDim.x) {
        float v = 0.0f;
        // first Linear: rows (W1[n][:], b1[n], 0..)
        if (i >= lay.w1 && i < lay.w1 + (int64_t)TCW * lay.O4) {
            const int n = (int)((i - lay.w1) / lay.O4), o = (int)((i - lay.w1) % lay.O4);
            const float *Wf = params + lay.flat_w[0];
            if (o < lay.O) v = Wf[(int64_t)n * lay.O + o];
            else if (o == lay.O) v = Wf[(int64_t)TCW * lay.O + n];
        } else if (i >= lay.wo && i < lay.wo + (int64_t)lay.A * TCW) {
            v = params[lay.flat_w[nl - 1] + (i - lay.wo)];
        } else if (i >= lay.bo && i < lay.bo + lay.A) {
            v = params[lay.flat_w[nl - 1] + (int64_t)lay.A * TCW + (i - lay.bo)];
        } else {
            for (int l = 1; l < nl - 1; ++l) {
                const float *Wf = params + lay.flat_w[l];   // [N][K] torch layout = K-major B operand
                if (i >= lay.bias[l] && i < lay.bias[l] + TCW) v = Wf[(int64_t)TCW * TCW + (i - lay.bias[l])];
                const bool hi = i >= lay.whi[l] && i < lay.whi[l] + TCW * TCW;
                const bool lo = i >= lay.wlo[l] && i < lay.wlo[l] + TCW * TCW;
                if (hi || lo) {                             // K-major core-matrix layout, rows n, cols k
                    int n, k;
                    core_invert(TCW, i - (hi ? lay.whi[l] : lay.wlo[l]), &n, &k);
                    const float w = Wf[(int64_t)n * TCW + k];
                    const float whi = tf32_hi(w);
                    v = hi ? whi : (w - whi);
                }
                const bool bhi = lay.wbhi[l] >= 0 && i >= lay.wbhi[l] && i < lay.wbhi[l] + TCW * TCW;
                const bool blo = lay.wblo[l] >= 0 && i >= lay.wblo[l] && i < lay.wblo[l] + TCW * TCW;
                if (bhi || blo) {                           // MN-major SW128_32B layout, rows n, cols k
                    int n, k;
                    mn32_invert(TCW, i - (bhi ? lay.wbhi[l] : lay.wblo[l]), &n, &k);
                    const float w = Wf[(int64_t)n * TCW + k];
                    const float whi = tf32_hi(w);
                    v = bhi ? whi : (w - whi);
                }
            }
        }
        packed[i] = v;
    }
}

int tg_pack_weights_tc(tg_ctx *ctx, const tg_tc_layout &lay, const float *params, cudaStream_t st) {
    int rc = tg_ctx_grow(ctx, (void **)&ctx->packed_tc, &ctx->packed_tc_cap, (size_t)lay.total * sizeof(float));
    if (rc) return rc;
    int64_t blocks = (lay.total + 255) / 256;
    if (blocks > 1024) blocks = 1024;
    pack_tc_kernel<<<(unsigned)blocks, 256, 0, st>>>(lay, params, ctx->packed_tc);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

// ---------------------------------------------------------------------------
// wide tensor-core staging (TcwLayout, tg_common.cuh)
// ---------------------------------------------------------------------------
void tg_build_tcw_layout(const tg_mlp_cfg *mlp, TcwLayout *L, bool with_backward) {
    memset(L, 0, sizeof(*L));
    L->O = mlp->dims[0];
    L->OKP = (L->O + 1 + 7) / 8 * 8;
    L->A = mlp->dims[3];
    L->act = mlp->activation;
    L->W = mlp->dims[1];
    const int W = L->W;
    int64_t off = 0;
    L->w0hi = off; off += (int64_t)W * L->OKP;
    L->w0lo = off; off += (int64_t)W * L->OKP;
    L->b1 = off; off += W;
    L->wo = off; off += (int64_t)L->A * W;
    L->bo = off; off += 4;
    L->resident = (off + 255) / 256 * 256;
    L->chunk_floats = (int64_t)W * 32;
    L->chunks_f = L->resident;
    L->chunks_b = L->chunks_f + (int64_t)(2 * W / 32) * L->chunk_floats;
    L->total = with_backward ? L->chunks_b + (int64_t)(2 * W / 32) * L->chunk_floats : L->chunks_b;
    int64_t flat = 0;
    for (int l = 0; l < 3; ++l) {
        L->flat_w[l] = flat;
        flat += (int64_t)mlp->dims[l] * mlp->dims[l + 1] + mlp->dims[l + 1];
    }
    L->n_params = flat;
}

__global__ void pack_tcw_kernel(TcwLayout L, const float *__restrict__ params, float *__restrict__ packed) {
    const int W = L.W;
    const float *W0 = params + L.flat_w[0], *b0 = W0 + (int64_t)W * L.O;
    const float *W1 = params + L.flat_w[1], *b1 = W1 + (int64_t)W * W;
    const float *Wo = params + L.flat_w[2], *bo = Wo + (int64_t)L.A * W;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < L.total; i += (int64_t)gridDim.x * blockDim.x) {
        float v = 0.0f;
        if (i < L.b1) {
            const bool lo = i >= L.w0lo;
            int n, c;
            core_invert(L.OKP, i - (lo ? L.w0lo : L.w0hi), &n, &c);
            const float w = c < L.O ? W0[(int64_t)n * L.O + c] : (c == L.O ? b0[n] : 0.0f);
            const float h = tf32_hi(w);
            v = lo ? (w - h) : h;
        } else if (i < L.wo) {
            v = b1[i - L.b1];
        } else if (i < L.bo) {
            v = Wo[i - L.wo];
        } else if (i < L.bo + L.A) {
            v = bo[i - L.bo];
        } else if (i >= L.chunks_f && i < L.chunks_b) {
            // forward: chunk = (K-chunk kc, hi/lo); [W rows n][32 k] K-major core-matrix layout
            const int64_t j = i - L.chunks_f;
            const int chunk = (int)(j / L.chunk_floats);
            const bool lo = (chunk & 1) != 0;
            const int kc = chunk >> 1;
            int n, kk;
            core_invert(32, j % L.chunk_floats, &n, &kk);
            const float w = W1[(int64_t)n * W + kc * 32 + kk];
            const float h = tf32_hi(w);
            v = lo ? (w - h) : h;
        } else if (i >= L.chunks_b) {
            // backward: chunk = (32 out-rows kc, hi/lo); [32 rows out][W cols in] MN-major SW128_32B layout
            const int64_t j = i - L.chunks_b;
            const int chunk = (int)(j / L.chunk_floats);
            const bool lo = (chunk & 1) != 0;
            const int kc = chunk >> 1;
            int r, c;
            mn32_invert(32, j % L.chunk_floats, &r, &c);
            const float w = W1[(int64_t)(kc * 32 + r) * W + c];
            const float h = tf32_hi(w);
            v = lo ? (w - h) : h;
        }
        packed[i] = v;
    }
}

int tg_pack_weights_tcw(tg_ctx *ctx, const TcwLayout &lay, const float *params, cudaStream_t st) {
    int rc = tg_ctx_grow(ctx, (void **)&ctx->packed_tc, &ctx->packed_tc_cap, (size_t)lay.total * sizeof(float));
    if (rc) return rc;
    pack_tcw_kernel<<<296, 256, 0, st>>>(lay, params, ctx->packed_tc);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

extern "C" int tg_ctx_sm_count(const tg_ctx *ctx) { return ctx ? ctx->sm_count : 0; }

int tg_ctx_grow(tg_ctx *ctx, void **buf, size_t *cap, size_t bytes) {
    if (bytes <= *cap) return TG_OK;
    TG_CUDA(cudaSetDevice(ctx->device));
    if (*buf) {
        TG_CUDA(cudaDeviceSynchronize());
        TG_CUDA(cudaFree(*buf));
        *buf = nullptr;
        *cap = 0;
    }
    TG_CUDA(cudaMalloc(buf, bytes));
    *cap = bytes;
    return TG_OK;
}

int tg_gauss_consts(const float *cov_diag, int A, float *sd, float *inv_sd, float *inv_var, float *log_norm) {
    double ln = 0.5 * A * log(2.0 * M_PI);
    for (int j = 0; j < A; ++j) {
        TG_REQUIRE(cov_diag[j] > 0.0f, TG_ERR_ARG, "cov_diag[%d] must be positive", j);
        const float s = sqrtf(cov_diag[j]);
        if (sd) sd[j] = s;
        if (inv_sd) inv_sd[j] = 1.0f / s;
        if (inv_var) inv_var[j] = 1.0f / (s * s);
        ln += (double)logf(s);
    }
    *log_norm = (float)ln;
    return TG_OK;
}

extern "C" int tg_env_dims(int kind, int *obs_dim, int *act_dim) {
    static const int O[4] = {5, 3, 10, 20}, A[4] = {1, 1, 2, 4};
    if (kind < 0 || kind > 3) {
        tg_set_error("unknown env kind %d", kind);
        return TG_ERR_ARG;
    }
    if (obs_dim) *obs_dim = O[kind];
    if (act_dim) *act_dim = A[kind];
    return TG_OK;
}

extern "C" int64_t tg_mlp_param_count(const tg_mlp_cfg *mlp) {
    if (!mlp || mlp->n_layers < 1 || mlp->n_layers > TG_MAX_LAYERS) return -1;
    int64_t n = 0;
    for (int l = 0; l < mlp->n_layers; ++l) n += (int64_t)mlp->dims[l] * mlp->dims[l + 1] + mlp->dims[l + 1];
    return n;
}

// FP32 FMA-pipe microbenchmark: MEASURED_PEAKS.json holds no FP32 peak, and the
// register-tiled MLP GEMMs are bounded by exactly this pipe.  16 independent FFMA
// chains per thread, 8 warps x 4 CTAs per SM.
__global__ void __launch_bounds__(256) fma_peak_kernel(int iters, float *sink) {
    float a[16];
    const float x = 1.0f + 1e-7f * threadIdx.x, y = 1e-3f * blockIdx.x;
#pragma unroll
    for (int i = 0; i < 16; ++i) a[i] = (float)i;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 16; ++i) a[i] = fmaf(a[i], x, y);
    }
    float s = 0.0f;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += a[i];
    if (s == 123.456f) sink[0] = s;
}

extern "C" int tg_fp32_peak(tg_ctx *ctx, double *out_tflops) {
    TG_REQUIRE(ctx && out_tflops, TG_ERR_ARG, "tg_fp32_peak: null argument");
    TG_CUDA(cudaSetDevice(ctx->device));
    float *sink = nullptr;
    TG_CUDA(cudaMalloc(&sink, 64));
    cudaEvent_t e0, e1;
    TG_CUDA(cudaEventCreate(&e0));
    TG_CUDA(cudaEventCreate(&e1));
    const int iters = 20000, grid = ctx->sm_count * 8;
    double best = 0.0;
    for (int rep = 0; rep < 6; ++rep) {
        TG_CUDA(cudaEventRecord(e0));
        fma_peak_kernel<<<grid, 256>>>(iters, sink);
        TG_CUDA(cudaEventRecord(e1));
        TG_CUDA(cudaEventSynchronize(e1));
        float ms = 0.0f;
        TG_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        const double fl = 2.0 * 16.0 * iters * 256.0 * grid;
        const double tf = fl / (ms * 1e-3) / 1e12;
        if (rep > 0 && tf > best) best = tf;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(sink);
    *out_tflops = best;
    return TG_OK;
}

size_t tg_update_smem_bytes(const tg_mlp_layout &lay, bool with_weights) {
    const int B = lay.B, NT = lay.NT, LDX = B + 4;
    size_t fl = (size_t)tg_round_up(lay.O, 8) * LDX + (size_t)(lay.n_layers - 1) * lay.NP * LDX + 8 * LDX +
                (size_t)(NT / B) * TG_MAX_ACT * B;
    if (with_weights) fl += (size_t)lay.total;
    return fl * sizeof(float);
}

int tg_build_layout(const tg_mlp_cfg *mlp, bool with_backward, tg_mlp_layout *out, int smem_limit) {
    TG_REQUIRE(mlp != nullptr, TG_ERR_ARG, "mlp cfg is null");
    TG_REQUIRE(mlp->n_layers >= 1 && mlp->n_layers <= TG_MAX_LAYERS, TG_ERR_SHAPE, "n_layers %d not in [1,%d]",
               mlp->n_layers, TG_MAX_LAYERS);
    TG_REQUIRE(mlp->activation >= TG_ACT_PER_LAYER && mlp->activation <= 2, TG_ERR_ARG, "unknown activation %d",
               mlp->activation);
    const int nl = mlp->n_layers;
    if (mlp->activation == TG_ACT_PER_LAYER)
        for (int l = 0; l < nl - 1; ++l)
            TG_REQUIRE(mlp->layer_activation[l] >= 0 && mlp->layer_activation[l] <= 2, TG_ERR_ARG,
                       "unknown activation %d after hidden layer %d", mlp->layer_activation[l], l);
    TG_REQUIRE(mlp->dims[0] >= 1 && mlp->dims[0] <= TG_MAX_WIDTH, TG_ERR_SHAPE, "input dim %d out of range", mlp->dims[0]);
    TG_REQUIRE(mlp->dims[nl] >= 1 && mlp->dims[nl] <= TG_MAX_ACT, TG_ERR_SHAPE, "output dim %d not in [1,%d]",
               mlp->dims[nl], TG_MAX_ACT);
    int maxh = 0, kmax = mlp->dims[0];
    for (int l = 1; l < nl; ++l) {
        TG_REQUIRE(mlp->dims[l] >= 1, TG_ERR_SHAPE, "hidden dim must be positive");
        maxh = mlp->dims[l] > maxh ? mlp->dims[l] : maxh;
        kmax = mlp->dims[l] > kmax ? mlp->dims[l] : kmax;
    }
    TG_REQUIRE(maxh <= TG_MAX_WIDTH, TG_ERR_UNSUPPORTED, "hidden width %d > %d is not supported", maxh, TG_MAX_WIDTH);
    memset(out, 0, sizeof(*out));
    out->n_layers = nl;
    out->act = mlp->activation;
    for (int l = 0; l < TG_MAX_LAYERS; ++l)
        out->acts[l] = mlp->activation == TG_ACT_PER_LAYER ? (l < nl - 1 ? mlp->layer_activation[l] : 0) : mlp->activation;
    out->cfg = maxh <= 64 ? 0 : (maxh <= 128 ? 1 : 2);
    out->O = mlp->dims[0];
    out->A = mlp->dims[nl];
    for (;;) {
        static const int Bs[4] = {128, 128, 64, 64}, NTs[4] = {128, 256, 256, 128}, NPs[4] = {64, 128, 256, 128};
        out->B = Bs[out->cfg];
        out->NT = NTs[out->cfg];
        out->NP = NPs[out->cfg];
        if (smem_limit <= 0 || out->cfg != 1) break;
        // deep width-128 nets (e.g. the reference's CartPole 128^4): the B=128 activation tiles of
        // the update kernel do not fit -> halve the sample tile
        if (tg_update_smem_bytes(*out, false) <= (size_t)smem_limit) break;
        out->cfg = 3;
    }
    // hidden outputs are stored for NP (padded) neurons, so the buffers need NP rows
    out->kmax = nl > 1 ? (out->NP > kmax ? out->NP : kmax) : kmax;
    int64_t off = 0, flat = 0;
    for (int l = 0; l < nl; ++l) {
        tg_layer_layout &L = out->L[l];
        L.K = mlp->dims[l];
        L.N = mlp->dims[l + 1];
        L.flat_w = flat;
        flat += (int64_t)L.K * L.N + L.N;
        L.wn = -1;
        L.KP = out->NP;
        if (l < nl - 1) {
            L.wt = off; off += (int64_t)L.K * out->NP;
            L.bias = off; off += out->NP;
            if (with_backward && l >= 1) { L.wn = off; off += (int64_t)L.N * out->NP; }
        } else {
            L.wt = off; off += tg_round_up(L.N * L.K, 4);
            L.bias = off; off += 4;
        }
    }
    out->total = off;
    out->n_params = flat;
    return TG_OK;
}

__global__ void pack_kernel(tg_mlp_layout lay, const float *__restrict__ params, float *__restrict__ packed) {
    const int nl = lay.n_layers, NP = lay.NP;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < lay.total;
         i += (int64_t)gridDim.x * blockDim.x) {
        float v = 0.0f;
        for (int l = 0; l < nl; ++l) {
            const tg_layer_layout &L = lay.L[l];
            const float *Wf = params + L.flat_w;          // [N][K] torch layout
            const float *bf = Wf + (int64_t)L.N * L.K;
            if (l < nl - 1) {
                if (i >= L.wt && i < L.wt + (int64_t)L.K * NP) {
                    const int k = (int)((i - L.wt) / NP), n = (int)((i - L.wt) % NP);
                    v = n < L.N ? Wf[(int64_t)n * L.K + k] : 0.0f;
                } else if (i >= L.bias && i < L.bias + NP) {
                    const int n = (int)(i - L.bias);
                    v = n < L.N ? bf[n] : 0.0f;
                } else if (L.wn >= 0 && i >= L.wn && i < L.wn + (int64_t)L.N * NP) {
                    const int n = (int)((i - L.wn) / NP), k = (int)((i - L.wn) % NP);
                    v = k < L.K ? Wf[(int64_t)n * L.K + k] : 0.0f;
                }
            } else {
                if (i >= L.wt && i < L.wt + (int64_t)L.N * L.K) v = Wf[i - L.wt];
                else if (i >= L.bias && i < L.bias + L.N) v = bf[i - L.bias];
            }
        }
        packed[i] = v;
    }
}

int tg_pack_weights(tg_ctx *ctx, const tg_mlp_layout &lay, const float *params, cudaStream_t st) {
    int rc = tg_ctx_grow(ctx, (void **)&ctx->packed, &ctx->packed_cap, (size_t)lay.total * sizeof(float));
    if (rc) return rc;
    const int threads = 256;
    int64_t blocks = (lay.total + threads - 1) / threads;
    if (blocks > 1024) blocks = 1024;
    pack_kernel<<<(unsigned)blocks, threads, 0, st>>>(lay, params, ctx->packed);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}
