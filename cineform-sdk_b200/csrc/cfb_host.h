// cfb_host.h -- host-side internals shared by the C-ABI translation units.
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <cstring>
#include <string>

#include "../../include/cfhd_b200.h"
#include "cfb_common.cuh"

namespace cfb {

void set_error(const char *fmt, ...);
cfb_error cuda_fail(cudaError_t e, const char *what);

#define CFB_CUDA(call)                                                  \
    do {                                                                \
        cudaError_t e_ = (call);                                        \
        if (e_ != cudaSuccess) return ::cfb::cuda_fail(e_, #call);      \
    } while (0)

QuantParam make_quant_param(int divisor, int midpoint_prequant, bool plain_midpoint = false);
// wait for everything queued on the context's stream without busy-waiting on a CPU core
cudaError_t stream_wait(cfb_context *ctx);

// kernel launchers (cfb_forward.cu / cfb_inverse.cu)
cudaError_t launch_fwd_plane(const FwdParams &p, int prescale, cudaStream_t stream);
cudaError_t launch_fwd_422(const FwdParams &p, cudaStream_t stream);
cudaError_t launch_fwd_rg48(const FwdParams &p, int sel, cudaStream_t stream);
cudaError_t launch_fwd_rg48_all(const FwdParams &p, cudaStream_t stream);
cudaError_t launch_fwd_byr4(const FwdParams &p, cudaStream_t stream);
cudaError_t launch_fwd_rgb30(const FwdParams &p, cudaStream_t stream);
cudaError_t launch_inv_plane(const InvParams &p, int descale, cudaStream_t stream);
// out: kInv422Out8 (YUYV / UYVY), kInv422OutYU64, kInv422OutV210 (cfb_common.cuh)
cudaError_t launch_inv_422(const InvParams &p, int out, cudaStream_t stream);
cudaError_t launch_inv_444_rg48(const InvParams &p, int out, cudaStream_t stream);
cudaError_t launch_lowpass_422(const InvParams &p, cudaStream_t stream);
cudaError_t launch_inv_fields(const InvParams &p, const FieldsAux &a, bool planar, cudaStream_t stream);
cudaError_t launch_fwd_422_fields(const FwdParams &p, cudaStream_t stream);
cudaError_t launch_fwd_422_fields_src(const FwdParams &p, int sel, cudaStream_t stream);
cudaError_t launch_fwd_yu64(const FwdParams &p, cudaStream_t stream);
// range audit of the planes a forward level is about to read (cfb_audit.cu): ORs violation bits into ctx->d_range
cfb_error audit_level_input(cfb_context *ctx, const FwdParams &p, int prescale);
cfb_error range_status(cfb_context *ctx, int *flags);
cudaError_t launch_fwd_v210(const FwdParams &p, cudaStream_t stream);

// The host forms of the transform as three stages, each on a stream of the caller's choice, so that the frame pool can
// run uploads, kernels and downloads of different jobs on separate streams (copy engines + SMs all busy).  The compute
// stage always runs on cfb_context_stream(); the caller orders the stages with events.  Slots [0, n) of the codec's
// device staging are used.  The synchronous C-ABI calls are these three stages on one stream + a wait.
cfb_error stage_fwd_upload(cfb_codec *cd, int n, const void *const *h_frames, int frame_pitch, cudaStream_t s);
cfb_error stage_fwd_compute(cfb_codec *cd, int n, const cfb_quant *quant, bool sparse);
// sparse: copies the first `guess` bytes of every frame's sparse buffer (speculative single pass); dense: the coded region
cfb_error stage_fwd_download(cfb_codec *cd, int n, void *const *h_out, bool sparse, unsigned guess, cudaStream_t s);
// sparse only, after the download has completed: fetches the bytes beyond `guess` (if any frame has more), reports sizes
cfb_error stage_fwd_tail(cfb_codec *cd, int n, void *const *h_sparse, unsigned guess, cudaStream_t s, size_t *sizes,
                         unsigned *max_bytes, bool *more);
cfb_error stage_inv_upload(cfb_codec *cd, int n, const void *const *h_in, bool sparse, cudaStream_t s);
cfb_error stage_inv_compute(cfb_codec *cd, int n, const cfb_quant *quant, int out_format, bool sparse);
cfb_error stage_inv_download(cfb_codec *cd, int n, void *const *h_frames, int frame_pitch, int out_format, cudaStream_t s);
unsigned sparse_initial_guess(const cfb_codec *cd);
unsigned sparse_next_guess(const cfb_codec *cd, unsigned max_bytes);
// GPU compaction / expansion between the pyramids and the sparse staging buffers of slots [0, n) (kernels only)
cfb_error sparse_upload(cfb_codec *cd, int n, const void *const *h_sparse, cudaStream_t s);
cfb_error sparse_download(cfb_codec *cd, int n, void *const *h_sparse, unsigned guess, cudaStream_t s);
cfb_error sparse_compact_device(cfb_codec *cd, int n);
cfb_error sparse_expand_device(cfb_codec *cd, int n);

}  // namespace cfb

struct cfb_context {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;             // blocking-sync event: host threads sleep instead of spinning
    int sm_count = 0;
    int *d_range = nullptr;                 // device flag word of the range audit (cfb_audit.cu), allocated on first use
    int *h_range = nullptr;                 // pinned copy
    std::atomic<uint64_t> kernel_launches{0}, frames_forward{0}, frames_inverse{0}, h2d_bytes{0}, d2h_bytes{0};
};

struct cfb_codec {
    cfb_context *ctx = nullptr;
    cfb_frame_desc desc{};
    cfb_layout layout{};
    int max_batch = 0;
    unsigned char *d_frames = nullptr;      // max_batch packed frames
    unsigned char *d_pyramids = nullptr;    // max_batch pyramids
    size_t frame_stride = 0;                // bytes between device frame slots
    size_t pyramid_stride = 0;
    int bayer_phase = 0;                    // BAYER_FORMAT_* (0 RED_GRN, 1 GRN_RED, 2 GRN_BLU, 3 BLU_GRN), DemoasicFrames.h:30
    int fwd_mask = 7, inv_mask = 7;         // profiling aid: levels to run
    int interlaced = 0;                     // level 1 is the field transform (CFHD_ENCODING_FLAGS_YUV_INTERLACED)
    int *d_carry = nullptr;                 // interlaced inverse: HL row carries, kMaxBatch frames
    unsigned short *d_curve = nullptr;      // Bayer encode curve (1 << 14 entries), null = frame already curved
    unsigned char *d_gop = nullptr;         // two-frame GOP buffer (cfb_gop2_layout.total_bytes), allocated on first use
    int carry_strips = 0;
    int decode_res = 1;                     // CFB_RESOLUTION_*: 1 full, 2 half (LL1), 3 quarter (LL2)
    // sparse transfer format staging (allocated on first use)
    unsigned char *d_sparse = nullptr;      // max_batch sparse buffers
    unsigned long long *d_status = nullptr; // max_batch * (nblocks + 1): look-back state of the one-pass packer
    unsigned *h_headers = nullptr;          // pinned, 4 u32 per slot
    size_t sparse_stride = 0;
    // B64A output (8 bytes per pixel) does not fit the frame staging of a 6-byte-per-pixel source: own staging, allocated on first use
    unsigned char *d_out64 = nullptr;
    size_t out64_stride = 0;
    unsigned value_guess = 0;               // running estimate of a frame's sparse size in bytes (speculative single-pass D2H)
};
