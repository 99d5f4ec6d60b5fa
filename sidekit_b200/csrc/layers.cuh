// Host-side launch wrappers for the kernels in layers.cu / frontend.cu / conv_umma.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace skb {

struct ConvParams;

struct FrontendConsts {
    int n_fft = 0, win = 0, hop = 0, n_mels = 0, n_out = 0, n_w = 0;
    float preemph = 0.97f;         // PreEmphasis coefficient (sidekit/nnet/augmentation.py:59-74), read from the checkpoint's flipped_filter
    float* window = nullptr;
    float2* tw_half = nullptr;
    float2* tw_full = nullptr;
    int *mel_lo = nullptr, *mel_cnt = nullptr, *mel_ofs = nullptr;
    float* mel_w = nullptr;
    float* dct = nullptr;
};

struct StemConsts { float w[128 * 9]; float b[128]; };   // folded stem conv + BN (<= 128 channels), passed to the kernel by value
int launch_stem(bool bf16, int cout, const float* feats, const long long* feat_off, const int* n_frames, const float2* cmvn,
                const StemConsts& sc, uint16_t* out, long long out_plane, int G, int p_end, int Wp, int W,
                const int* row_b, const int* row_h, unsigned* overflow, cudaStream_t st);
int launch_stem7(bool bf16, const float* feats, const long long* feat_off, const int* n_frames, const float2* cmvn,
                 const StemConsts& sc, uint16_t* out, long long out_plane, int G, int p_end, int Wp, int W, int F,
                 const int* row_b, const int* row_h, unsigned* overflow, cudaStream_t st);
int launch_broadcast_rows(const float* bias, int B, int A, float* out, cudaStream_t st);
struct PlaneSumArgs { int p_end; const int* pix_b; const int* span_b; };   // launch_se_scale: channel totals beside the border sums
int span_table_size(int n_pix);
int launch_span_table(const int* pix_b, int n_pix, int* span_b, cudaStream_t st);
int launch_se_scale(bool bf16, unsigned long long* sums, const uint16_t* y1, long long plane, int G, int Wp, int W,
                    const int* utt_row0, const int* utt_count, int B, int Cin, int Cout, const float* w2t, const float* b2,
                    const float* fc1, const float* fc2, float* brd_ws, float* scale, cudaStream_t st,
                    const PlaneSumArgs* totals = nullptr);
int launch_gather_frames(bool bf16, const uint16_t* act, long long plane, int C, int W, int Wp, int G,
                         const int* frame_row, int n_frames, uint16_t* X, cudaStream_t st);
int launch_gather_pack(const uint16_t* act, long long plane, int C, int W, int Wp, int G, const int* frame_row, int n_frames,
                       uint16_t* hi, cudaStream_t st);
int launch_meanstd_planes(bool bf16, const uint16_t* act, long long plane, int G, const int* utt_row0, const int* n_fr, int B, int D,
                          const float* aff_s, const float* aff_t, float* out, cudaStream_t st);
int launch_meanstd(bool bf16, const uint16_t* X, const long long* frame_off, const int* n_fr, int B, int D, const float* aff_s,
                   const float* aff_t, float* out, cudaStream_t st);
int launch_att_act(float* h, const float* hb, const int* frame_utt, const float* bn_s, const float* bn_t, int n_frames,
                   int A, cudaStream_t st);
int launch_softmax_pool(bool bf16, const uint16_t* X, const float* logit, const long long* frame_off, const int* n_fr, int B, int D,
                        float* out, cudaStream_t st);
int launch_head_norm(const float* x, const float* aff_s, const float* aff_t, int B, int E, int norm_embedding,
                     float* emb_pre, float* emb, cudaStream_t st);
int launch_sgemm_nt(const float* A, const float* B, float* C, const float* bias, int M, int N, int K, int lda, int ldb,
                    int ldc, float alpha, cudaStream_t st);
size_t skinny_gemm_ws_floats(int M, int N, int K);
int launch_skinny_gemm(const float* A, int M, int K, const float* W, int N, const float* bias, float alpha, float* C, int ldc,
                       float* ws, cudaStream_t st);
int launch_pack_frames(bool bf16, const float* X, int C_src, int C_dst, int n_rows, const int* row_src, const int* row_b,
                       const float2* cmvn, uint16_t* out, long long plane, int G, cudaStream_t st);

// scoring.cu: split-precision tcgen05 GEMM on packed fp16 operands (also used for the dense layers of the extractor)
struct TrialTables;
struct PackedOp {
    uint16_t* hi = nullptr;      // [rows_pad/128][Dp/8][128][8] fp16 high parts (lo follows in the same allocation)
    uint16_t* lo = nullptr;
    unsigned* stats = nullptr;   // device: max |x| bits, max row sum of squares bits, then the int scale exponent
    int* exp = nullptr;
    int rows = 0, rows_pad = 0, D = 0, Dp = 0;
};
int packed_create(const float* X_dev, int rows, int D, PackedOp* op, cudaStream_t st);
void packed_free(PackedOp* op);
int gemm_nt_split(const float* A_dev, int M, int K, const PackedOp& W, const float* bias, float alpha, float* C, int ldc,
                  cudaStream_t st);
// same with an A operand that is already packed (hi planes written by the caller, lo planes zero, scale exponent 0)
int packed_alloc_zero(PackedOp* op, int rows, int D, cudaStream_t st);
int gemm_workspace_reserve(int M, int K);
int gemm_packed_a(const PackedOp& A, const PackedOp& W, const float* bias, float alpha, float* C, int ldc, cudaStream_t st);

// conv_umma.cu
int launch_conv_umma(const ConvParams& p, int n_cta, bool bf16, cudaStream_t st);
int conv_tile_m(int n_cta);          // output pixels per CTA for a given N_CTA configuration
int conv_pick_ncta(int cout);        // 32 / 64 / 128
bool conv_sums_supported(int n_cta, int cout);   // can an unfused conv's epilogue accumulate the SE channel totals (ConvParams::sums)

// frontend.cu
int frontend_consts_create(FrontendConsts* fc, int n_fft, int win, int hop, int n_mels, int n_out, const float* window,
                           const float* fb, const float* dct);
void frontend_consts_destroy(FrontendConsts* fc);
// Writes raw features (frame-major) and the per-(utterance, coefficient) CMVN statistics (mean, rstd) into `cmvn`
// ([B][n_out] float2; `cmvn_part` is scratch of frontend_cmvn_scratch_bytes()).  With `normalise` the features are
// also normalised in place (and optionally written as the (B, n_out, t_max) tensor the reference's front-end returns);
// without it the consumer (the stem kernel) applies the statistics on the fly.
int frontend_launch(const FrontendConsts& fc, const float* wave, const long long* wave_off, const int* wave_len,
                    const long long* feat_off, const int* n_frames, int B, int t_max, float* feats, float2* cmvn,
                    void* cmvn_part, bool normalise, float* api_out, cudaStream_t stream);
size_t frontend_cmvn_scratch_bytes(const FrontendConsts& fc, int B, int t_max);

}  // namespace skb
