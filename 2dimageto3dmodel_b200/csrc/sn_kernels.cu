// Weight bank: spectral normalisation + kernel weight layouts for ALL convolutions of a network in a handful of
// launches (SURVEY.md §2.2 "spectral norm power iteration ... per layer per forward"; VERDICT r1 "weak" #6: ~1 000
// tiny cuBLAS gemv / dot / elementwise launches per step and per-call permute+contiguous weight re-layouts).
//
// Reference semantics: torch.nn.utils.spectral_norm as the reference applies it (models/gan.py:57-65,163-177,294-302):
//   training:  v <- normalize(W^T u);  u <- normalize(W v);  sigma = u . (W v);  W_sn = W / sigma      (one power iteration,
//              u / v updated in place under no_grad, normalize(x) = x / max(|x|, 1e-12))
//   eval:      sigma = u . (W v) with the stored u, v
//   backward:  dW = (dW_sn - <dW_sn, W_sn> u v^T) / sigma        (u, v are constants of the graph, as in torch)
// with W = weight_orig viewed as [Cout, K = Cin*kh*kw].
//
// Layouts written for the convolution kernels (csrc/tc_conv.cu, thin_kernels.cu):
//   F [T'][Cout][Cin']   tap-major, K-major rows: fprop B operand, wgrad output layout
//   D [T'][Cin'][Cout']  per-tap transpose (Cout' = Cout rounded up to 32, zero filled): dgrad B operand
// plain (fold = 0): T' = kh*kw, Cin' = Cin rounded up to 32 (zero filled);
// folded stems (fold = 1, discriminator conv1 with 8 / 11 input channels): the kh vertical taps live in the channel
// dimension, T' = kw, Cin' = kh*Cin rounded up to 32, F[s][co][r*Cin + c] = W[co][c][r][s] (b3d/conv.py:fold_kh_weight).
// up2 layers (3x3 convolutions whose input is a x2 nearest upsample, read before the upsample): ALSO the 16 taps of the four
// output-parity classes, UF [16][Cout][Cin'] and UD [16][Cin'][Cout'], tap ((a*2 + b)*2 + u)*2 + v = K_ab[u][v] with
// K_ab = A_a W A_b^T, A_0 = [[1,0,0],[0,1,1]], A_1 = [[1,1,0],[0,0,1]]: output pixel (2i+a, 2j+b) of conv3x3(up2(x)) is the
// 2x2 convolution K_ab of x at rows i+a-1+u, columns j+b+v (b3d/conv.py upconv_taps).  Summed in fp32 from W / sigma, then
// rounded to tf32 once.  The weight gradient still arrives in the 3x3 F layout (b3d_bank_up2_grad applies the adjoint).
//
// Launch structure: every kernel walks a host-built list of (layer, chunk) work items, one CTA each, so all layers of a
// network share the launches: zero scratch (memset) -> W^T u -> W v -> emit;  backward: <dF, F> -> dW.
#include "b3d_common.cuh"

namespace {

constexpr int NT = 256;
constexpr float SN_EPS = 1e-12f;

// Parameters (w, u, v) are addressed by pointer (they are the module's own tensors); everything a call produces is
// addressed by OFFSET (in floats) into per-call flat buffers passed as kernel arguments, so that two forward passes of
// the same network never alias (torch's spectral_norm clones u / v for the graph for the same reason).
struct alignas(16) BankLayer {
    const float* w;      // weight_orig [Cout][Cin][kh][kw]
    float* u;            // [Cout]   (spectral norm only; updated in place in training mode)
    float* v;            // [K]
    long long t_off;     // scratch [2K floats = K int64]: W^T u in 2^-36 fixed point (scratch is zeroed before the forward)
    long long s_off;     // scratch [Cout]: W v (/ |t|)
    long long wf_off;    // out: F layout
    long long wd_off;    // out: D layout, or -1
    long long u_off;     // out: u used by this call's graph [Cout]
    long long v_off;     // out: v used by this call's graph [K]
    long long scal_off;  // out: [2] = (sigma, <dF, F> accumulator)
    long long df_off;    // backward in : gradient in F layout (offset into the dF buffer = wf_off's numbering)
    long long dw_off;    // backward out: gradient in weight_orig layout
    long long uf_off;    // out: up2 class taps, UF layout, or -1
    long long ud_off;    // out: up2 class taps, UD layout, or -1
    int Cout, Cin, kh, kw;
    int fold, Cinp, Coutp, Tp;
    int sn, up2, pad1, pad2;
};

// the 16 class taps of a 3x3 kernel w[r][s] (see the layout comment at the top)
__device__ __forceinline__ void up2_taps(const float w[9], float k[16]) {
    float rw[2][2][3];                                  // rw[a][u][s] = sum_r A_a[u][r] w[r][s]
#pragma unroll
    for (int s = 0; s < 3; ++s) {
        rw[0][0][s] = w[s];
        rw[0][1][s] = w[3 + s] + w[6 + s];
        rw[1][0][s] = w[s] + w[3 + s];
        rw[1][1][s] = w[6 + s];
    }
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const float* q = rw[a][u];
            const float c[2][2] = {{q[0], q[1] + q[2]}, {q[0] + q[1], q[2]}};      // c[b][v] = sum_s A_b[v][s] q[s]
#pragma unroll
            for (int b = 0; b < 2; ++b)
#pragma unroll
                for (int v = 0; v < 2; ++v) k[((a * 2 + b) * 2 + u) * 2 + v] = c[b][v];
        }
}

struct Item { int layer, a, b, c; };

// W^T u is summed over row chunks by different CTAs.  fp32 atomics would make the sum depend on the arrival order (and with
// the tf32 rounding of the emitted weights a last-bit difference becomes a 2^-11 one: the same step would not repeat
// bit-for-bit), so the partial sums are accumulated as 64-bit integers in units of 2^-36: integer addition is associative,
// the result is the same whatever the order (resolution 1.5e-11, range +-1.3e8; |t| <= sigma_max(W), a few tens at most).
constexpr double T_SCALE = 68719476736.0;
__device__ __forceinline__ float t_value(const float* scratch, long long t_off, int k) {
    return (float)((double)reinterpret_cast<const long long*>(scratch + t_off)[k] * (1.0 / T_SCALE));
}

__device__ __forceinline__ float block_reduce_sum(float v, float* red) {
    v = b3d::warp_sum(v);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) red[w] = v;
    __syncthreads();
    float r = 0.f;
#pragma unroll
    for (int i = 0; i < NT / 32; ++i) r += red[i];
    return r;                       // every thread holds the block sum
}

// t[col] += sum_{rows of the chunk} W[row][col] * u[row]          item: (layer, column chunk of NT, row chunk of 64)
__global__ void __launch_bounds__(NT)
bank_wtu_kernel(const BankLayer* __restrict__ layers, const Item* __restrict__ items, float* __restrict__ scratch) {
    const Item it = items[blockIdx.x];
    const BankLayer L = layers[it.layer];
    const int K = L.Cin * L.kh * L.kw;
    const int col = it.a * NT + threadIdx.x;
    const int r0 = it.b * 64, r1 = min(r0 + 64, L.Cout);
    if (col >= K) return;
    float acc = 0.f;
    const float* w = L.w + (size_t)r0 * K + col;
#pragma unroll 8
    for (int r = r0; r < r1; ++r, w += K) acc = fmaf(__ldg(w), __ldg(L.u + r), acc);
    atomicAdd(reinterpret_cast<unsigned long long*>(scratch + L.t_off) + col,
              (unsigned long long)__double2ll_rn((double)acc * T_SCALE));
}

// training: s[row] = (W[row] . t) / max(|t|, eps)       eval: s[row] = W[row] . v         item: (layer, chunk of 8 rows)
__global__ void __launch_bounds__(NT)
bank_wv_kernel(const BankLayer* __restrict__ layers, const Item* __restrict__ items, float* __restrict__ scratch, int training) {
    __shared__ float red[NT / 32];
    const Item it = items[blockIdx.x];
    const BankLayer L = layers[it.layer];
    const int K = L.Cin * L.kh * L.kw;
    float inv = 1.f;
    if (training) {
        float p = 0.f;
        for (int k = threadIdx.x; k < K; k += NT) { const float x = t_value(scratch, L.t_off, k); p = fmaf(x, x, p); }
        inv = 1.f / fmaxf(sqrtf(block_reduce_sum(p, red)), SN_EPS);
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = it.a * (NT / 32) + warp;
    if (row >= L.Cout) return;
    const float* w = L.w + (size_t)row * K;
    float acc = 0.f;
    for (int k = lane; k < K; k += 32) acc = fmaf(__ldg(w + k), training ? t_value(scratch, L.t_off, k) : L.v[k], acc);
    acc = b3d::warp_sum(acc);
    if (lane == 0) scratch[L.s_off + row] = acc * inv;
}

// fp32 -> nearest tf32 value (ties away from zero), kept in an fp32 word: what the tensor core then reads exactly
__device__ __forceinline__ float tf32_rna(float x, int on) {
    if (!on) return x;
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}

__device__ __forceinline__ float layer_sigma(const BankLayer& L, const float* sv, int training, float* red, float* inv_s) {
    // training: u_new = s / max(|s|, eps), sigma = u_new . s;  eval: sigma = u . s
    float p = 0.f;
    for (int r = threadIdx.x; r < L.Cout; r += NT) {
        const float x = sv[r];
        p = fmaf(training ? x : L.u[r], x, p);
    }
    p = block_reduce_sum(p, red);
    if (!training) { *inv_s = 1.f; return p; }
    const float nrm = fmaxf(sqrtf(p), SN_EPS);
    *inv_s = 1.f / nrm;
    return p / nrm;
}

// Emit F (and D) for a (32 co) x (32 ci') chunk of all taps; chunk (0,0) also stores u, v, sigma.
// item: (layer, co chunk, ci' chunk)
__global__ void __launch_bounds__(NT)
bank_emit_kernel(const BankLayer* __restrict__ layers, const Item* __restrict__ items, const float* __restrict__ scratch,
                 float* __restrict__ outb, int training, int round_tf32) {
    __shared__ float red[NT / 32];
    const Item it = items[blockIdx.x];
    const BankLayer L = layers[it.layer];
    const int K = L.Cin * L.kh * L.kw, taps = L.kh * L.kw;
    float sigma = 1.f, inv_s = 1.f;
    if (L.sn) {
        const float* sv = scratch + L.s_off;
        sigma = layer_sigma(L, sv, training, red, &inv_s);
        if (it.a == 0 && it.b == 0) {       // one CTA per layer publishes u, v (in place + this call's copies) and sigma
            if (threadIdx.x == 0) { outb[L.scal_off] = sigma; outb[L.scal_off + 1] = 0.f; }
            float inv_t = 1.f;
            if (training) {
                float p = 0.f;
                for (int k = threadIdx.x; k < K; k += NT) { const float x = t_value(scratch, L.t_off, k); p = fmaf(x, x, p); }
                inv_t = 1.f / fmaxf(sqrtf(block_reduce_sum(p, red)), SN_EPS);
            }
            for (int k = threadIdx.x; k < K; k += NT) {
                const float x = training ? t_value(scratch, L.t_off, k) * inv_t : L.v[k];
                if (training) L.v[k] = x;
                outb[L.v_off + k] = x;
            }
            for (int r = threadIdx.x; r < L.Cout; r += NT) {
                const float x = training ? sv[r] * inv_s : L.u[r];
                if (training) L.u[r] = x;
                outb[L.u_off + r] = x;
            }
        }
    }
    const float rs = 1.f / sigma;
    const int co0 = it.a * 32, ci0 = it.b * 32;
    const int real_cin = L.fold ? L.kh * L.Cin : L.Cin;
    // F: lanes along ci' (coalesced stores), 8 co per pass
    for (int e = threadIdx.x; e < 32 * 32; e += NT) {
        const int ci = ci0 + (e & 31), co = co0 + (e >> 5);
        if (co >= L.Cout || ci >= L.Cinp) continue;
        const bool real = ci < real_cin;
        int c = ci, r_fix = 0;
        if (L.fold) { c = ci % L.Cin; r_fix = ci / L.Cin; }
        for (int tp = 0; tp < L.Tp; ++tp) {
            float val = 0.f;
            if (real) {
                const int src = L.fold ? ((co * L.Cin + c) * L.kh + r_fix) * L.kw + tp : (co * L.Cin + c) * taps + tp;
                val = tf32_rna(__ldg(L.w + src) * rs, round_tf32);
            }
            outb[L.wf_off + ((size_t)tp * L.Cout + co) * L.Cinp + ci] = val;
        }
    }
    if (L.up2) {
        // UF: lanes along ci' (coalesced stores)
        for (int e = threadIdx.x; e < 32 * 32; e += NT) {
            const int ci = ci0 + (e & 31), co = co0 + (e >> 5);
            if (co >= L.Cout || ci >= L.Cinp) continue;
            float w[9], k[16];
#pragma unroll
            for (int t = 0; t < 9; ++t) w[t] = ci < L.Cin ? __ldg(L.w + (co * L.Cin + ci) * 9 + t) * rs : 0.f;
            up2_taps(w, k);
#pragma unroll
            for (int t = 0; t < 16; ++t) outb[L.uf_off + ((size_t)t * L.Cout + co) * L.Cinp + ci] = tf32_rna(k[t], round_tf32);
        }
        // UD: lanes along co' (coalesced stores); rows co >= Cout are zero
        for (int e = threadIdx.x; e < 32 * 32; e += NT) {
            const int co = co0 + (e & 31), ci = ci0 + (e >> 5);
            if (co >= L.Coutp || ci >= L.Cinp) continue;
            float w[9], k[16];
#pragma unroll
            for (int t = 0; t < 9; ++t) w[t] = (ci < L.Cin && co < L.Cout) ? __ldg(L.w + (co * L.Cin + ci) * 9 + t) * rs : 0.f;
            up2_taps(w, k);
#pragma unroll
            for (int t = 0; t < 16; ++t) outb[L.ud_off + ((size_t)t * L.Cinp + ci) * L.Coutp + co] = tf32_rna(k[t], round_tf32);
        }
    }
    if (L.wd_off < 0) return;
    // D: lanes along co' (coalesced stores); rows co >= Cout are zero
    const int cop0 = it.a * 32;
    for (int e = threadIdx.x; e < 32 * 32; e += NT) {
        const int co = cop0 + (e & 31), ci = ci0 + (e >> 5);
        if (co >= L.Coutp || ci >= L.Cinp) continue;
        const bool real = ci < real_cin && co < L.Cout;
        int c = ci, r_fix = 0;
        if (L.fold) { c = ci % L.Cin; r_fix = ci / L.Cin; }
        for (int tp = 0; tp < L.Tp; ++tp) {
            float val = 0.f;
            if (real) {
                const int src = L.fold ? ((co * L.Cin + c) * L.kh + r_fix) * L.kw + tp : (co * L.Cin + c) * taps + tp;
                val = tf32_rna(__ldg(L.w + src) * rs, round_tf32);
            }
            outb[L.wd_off + ((size_t)tp * L.Cinp + ci) * L.Coutp + co] = val;
        }
    }
}

// <dF, F> per layer (spectral-norm layers only)        item: (layer, chunk of 4096 elements)
__global__ void __launch_bounds__(NT)
bank_bwd_dot_kernel(const BankLayer* __restrict__ layers, const Item* __restrict__ items, float* __restrict__ outb,
                    const float* __restrict__ dfb) {
    __shared__ float red[NT / 32];
    const Item it = items[blockIdx.x];
    const BankLayer L = layers[it.layer];
    if (!L.sn) return;
    const float* df = dfb + L.df_off;
    const float* wf = outb + L.wf_off;
    const size_t n = (size_t)L.Tp * L.Cout * L.Cinp;
    const size_t e0 = (size_t)it.a * 4096;
    float p = 0.f;
#pragma unroll 4
    for (int j = threadIdx.x; j < 4096; j += NT) {
        const size_t e = e0 + j;
        if (e < n) p = fmaf(__ldg(df + e), __ldg(wf + e), p);
    }
    p = block_reduce_sum(p, red);
    if (threadIdx.x == 0) atomicAdd(outb + L.scal_off + 1, p);
}

// dW[co][c][r][s] = (dF[...] - <dF,F> u[co] v[k]) / sigma          item: (layer, co chunk, ci' chunk)
__global__ void __launch_bounds__(NT)
bank_bwd_emit_kernel(const BankLayer* __restrict__ layers, const Item* __restrict__ items, const float* __restrict__ outb,
                     const float* __restrict__ dfb, float* __restrict__ dwb) {
    const Item it = items[blockIdx.x];
    const BankLayer L = layers[it.layer];
    const int taps = L.kh * L.kw, K = L.Cin * taps;
    const float sigma = L.sn ? outb[L.scal_off] : 1.f, ip = L.sn ? outb[L.scal_off + 1] : 0.f;
    const float* df = dfb + L.df_off;
    float* dw = dwb + L.dw_off;
    const float* uu = outb + L.u_off;
    const float* vv = outb + L.v_off;
    const float rs = 1.f / sigma;
    const int co0 = it.a * 32, ci0 = it.b * 32;
    const int real_cin = L.fold ? L.kh * L.Cin : L.Cin;
    for (int e = threadIdx.x; e < 32 * 32; e += NT) {
        const int ci = ci0 + (e & 31), co = co0 + (e >> 5);
        if (co >= L.Cout || ci >= real_cin) continue;
        int c = ci, r_fix = 0;
        if (L.fold) { c = ci % L.Cin; r_fix = ci / L.Cin; }
        const float uc = L.sn ? uu[co] * ip : 0.f;
        for (int tp = 0; tp < L.Tp; ++tp) {
            const int src = L.fold ? ((co * L.Cin + c) * L.kh + r_fix) * L.kw + tp : (co * L.Cin + c) * taps + tp;
            const float g = __ldg(df + ((size_t)tp * L.Cout + co) * L.Cinp + ci);
            dw[src] = L.sn ? (g - uc * vv[src - co * K]) * rs : g;
        }
    }
}

// Adjoint of the up2 class taps: dF[r*3 + s][co][ci] += sum_{R in {3-r, 2-r}} sum_{S in {3-s, 2-s}} dk[R*4 + S][ci][co], with dk
// the weight gradient of the up-convolution in b3d_conv2d_wgrad_tf32's tap-major layout [4x4][Cin][Cout] (tap (R, S) =
// class (a, b), tap (u, v) at R = 3 - a - 2u, S = 3 - b - 2v; b3d/conv.py _UpConvBanked).  One thread per (ci, co).
__global__ void __launch_bounds__(NT)
bank_up2_grad_kernel(const float* __restrict__ dk, float* __restrict__ df, int Cout, int Cin, int Cinp) {
    const long long e = (long long)blockIdx.x * NT + threadIdx.x;
    if (e >= (long long)Cin * Cout) return;
    const int co = (int)(e % Cout), ci = (int)(e / Cout);
    const size_t plane = (size_t)Cin * Cout;
    float g[16];
#pragma unroll
    for (int t = 0; t < 16; ++t) g[t] = __ldg(dk + t * plane + e);
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int s = 0; s < 3; ++s) {
            const int R = 3 - r, S = 3 - s;
            const float v = (g[R * 4 + S] + g[R * 4 + S - 1]) + (g[(R - 1) * 4 + S] + g[(R - 1) * 4 + S - 1]);
            df[((size_t)(r * 3 + s) * Cout + co) * Cinp + ci] += v;
        }
}

}  // namespace

extern "C" {

int b3d_bank_layer_bytes(void) { return (int)sizeof(BankLayer); }

// layers: device array of BankLayer records (b3d_bank_layer_bytes() each; the host packs them in the field order of the
// struct above); items_*: device arrays of int4 work items; scratch: per-bank device buffer (every layer's t / s,
// zeroed here); out: this call's flat output buffer (F / D layouts, u, v, sigma per layer).
// Enqueues: memset + W^T u (training only) + W v + emit.
int b3d_bank_forward(const void* layers, const void* items_wtu, int n_wtu, const void* items_wv, int n_wv,
                     const void* items_emit, int n_emit, float* scratch, size_t scratch_bytes, float* out, int training,
                     void* stream) {
    B3D_REQUIRE(layers && items_emit && scratch && out, B3D_EINVAL, "b3d_bank_forward: null pointer");
    B3D_REQUIRE(n_wv >= 0 && n_emit > 0 && n_wtu >= 0, B3D_EINVAL, "b3d_bank_forward: bad item counts");
    cudaStream_t st = (cudaStream_t)stream;
    B3D_CUDA_OK(cudaMemsetAsync(scratch, 0, scratch_bytes, st));
    const BankLayer* L = static_cast<const BankLayer*>(layers);
    const int flags = training;
    training &= 1;
    if (training && n_wtu > 0) {
        bank_wtu_kernel<<<n_wtu, NT, 0, st>>>(L, static_cast<const Item*>(items_wtu), scratch);
        B3D_LAUNCH_OK();
    }
    if (n_wv > 0) {
        bank_wv_kernel<<<n_wv, NT, 0, st>>>(L, static_cast<const Item*>(items_wv), scratch, training);
        B3D_LAUNCH_OK();
    }
    const int round_tf32 = (flags >> 1) & 1;          // bit 1 of `training`: round the emitted weights to tf32
    bank_emit_kernel<<<n_emit, NT, 0, st>>>(L, static_cast<const Item*>(items_emit), scratch, out, training, round_tf32);
    B3D_LAUNCH_OK();
    return B3D_OK;
}

// Gradients in F layout (df, numbered like the F region of `out`) -> gradients in weight_orig layout (dw); uses the u, v,
// sigma this call's forward stored in `out`.
int b3d_bank_backward(const void* layers, const void* items_dot, int n_dot, const void* items_emit, int n_emit, float* out,
                      const float* df, float* dw, void* stream) {
    B3D_REQUIRE(layers && items_emit && n_emit > 0 && n_dot >= 0 && out && df && dw, B3D_EINVAL, "b3d_bank_backward: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    const BankLayer* L = static_cast<const BankLayer*>(layers);
    if (n_dot > 0) {
        bank_bwd_dot_kernel<<<n_dot, NT, 0, st>>>(L, static_cast<const Item*>(items_dot), out, df);
        B3D_LAUNCH_OK();
    }
    bank_bwd_emit_kernel<<<n_emit, NT, 0, st>>>(L, static_cast<const Item*>(items_emit), out, df, dw);
    B3D_LAUNCH_OK();
    return B3D_OK;
}

// dk [16][Cin][Cout] (the up-convolution's weight gradient) -> ACCUMULATED into df [9][Cout][Cinp] (the layer's F-layout
// gradient sink)
int b3d_bank_up2_grad(const float* dk, float* df, int Cout, int Cin, int Cinp, void* stream) {
    B3D_REQUIRE(dk && df && Cout > 0 && Cin > 0 && Cinp >= Cin, B3D_EINVAL, "b3d_bank_up2_grad: bad arguments");
    const long long total = (long long)Cin * Cout;
    bank_up2_grad_kernel<<<(unsigned)((total + NT - 1) / NT), NT, 0, (cudaStream_t)stream>>>(dk, df, Cout, Cin, Cinp);
    B3D_LAUNCH_OK();
    return B3D_OK;
}

}  // extern "C"
