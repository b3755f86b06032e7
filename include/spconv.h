/*
 * spconv.h -- C ABI of libspconv.so: the B200 (sm_100a) spatial-parallel convolution engine
 * that sits under the torchgems Python API (mpi4dl_b200/torchgems/spatial.py).
 *
 * The reference (OSU-Nowlab/MPI4DL) has NO FFI: its hot path is Python calling
 * torch.nn.Conv2d / nn.AvgPool2d / nn.MaxPool2d / nn.ZeroPad2d and torch.distributed
 * (src/torchgems/spatial.py).  Each entry point below names the reference call site it
 * replaces.  Conventions (SURVEY.md section 8b):
 *   - plain pointers + sizes only; no torch / C++ types cross the boundary;
 *   - every pointer is a DEVICE pointer unless said otherwise; the caller owns all tensors;
 *   - all work is enqueued asynchronously on the given cudaStream_t (passed as void*);
 *   - return 0 on success, a negative SPC_E* code otherwise; spc_last_error() gives text;
 *   - not thread-safe per context (the reference is one host thread per process/GPU).
 *
 * Tensors are NCHW contiguous.  "Tile" = the part of the image owned by this rank
 * (train_spatial.py:241-290).  A tile's halo is delivered as up to 8 packed strips, indexed by
 * the reference's 3x3 neighbour stencil (spatial.py:961-964):   0 1 2 / 3 [4] 5 / 6 7 8
 *   strips 1,7 (top,bottom): [N][C][halo_h][W]     strips 3,5 (left,right): [N][C][H][halo_w]
 *   strips 0,2,6,8 (corners): [N][C][halo_h][halo_w]
 * exactly the message shapes of the reference (spatial.py:311-334 get_shapes_recv).  A NULL
 * strip means "no neighbour there": zeros are used (ZeroPad2d, spatial.py:142-144,1020).
 */
#ifndef SPCONV_H_
#define SPCONV_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPC_VERSION 100

enum { SPC_OK = 0, SPC_EINVAL = -1, SPC_ECUDA = -2, SPC_EUNSUPPORTED = -3, SPC_ENOMEM = -4 };
enum { SPC_F32 = 0, SPC_BF16 = 1 };             /* storage dtype of x / w / y; accumulation is fp32 */
enum { SPC_POOL_MAX = 0, SPC_POOL_AVG = 1 };
/* SPC_ALGO_TF32: like AUTO, but fp32 storage may use the tensor cores with TF32 operands (fp32 accumulate, fp32
 * output); with bf16 storage it is AUTO.  fp32 shapes the TF32 path does not cover, and the halo boundary rows /
 * columns of fp32 convolutions, run on the direct kernel in exact fp32.  With AUTO, fp32 is always exact fp32. */
enum { SPC_ALGO_AUTO = 0, SPC_ALGO_DIRECT = 1, SPC_ALGO_TCGEN05 = 2, SPC_ALGO_TF32 = 3 };

/* Geometry of one spatially-partitioned convolution on one tile.
 * Mirrors conv_spatial.__init__ (spatial.py:26-155): padding is "same"
 * (pad_h = (R-1)/2, pad_w = (S-1)/2, :115-121), dilation = 1, groups = 1 (:130-140). */
typedef struct {
  int32_t N, C, H, W;          /* input tile, unpadded */
  int32_t K, R, S;             /* filter [K][C][R][S] */
  int32_t stride_h, stride_w;
  int32_t pad_h, pad_w;        /* == halo_len_height / halo_len_width */
  int32_t dtype;               /* SPC_F32 | SPC_BF16 */
  int32_t algo;                /* SPC_ALGO_*; AUTO picks tcgen05 when the shape qualifies */
} spc_conv_desc;

typedef struct {
  int32_t N, C, H, W;
  int32_t k, stride, pad;      /* square window; pad == floor((k-1)/2) (spatial.py:1457-1464) */
  int32_t mode;                /* SPC_POOL_MAX | SPC_POOL_AVG */
  int32_t dtype;
} spc_pool_desc;

/* Received halo strips of a tile (device pointers, NULL = zero padding there). */
typedef struct {
  const void* strip[9];
} spc_halo;

/* ---- library / device ------------------------------------------------------------------- */
int         spc_version(void);
const char* spc_last_error(void);
/* sm count, compute capability major*10+minor; fails loudly when no sm_100 device is present */
int         spc_device_info(int device, int* sm_count, int* cc);
/* number of kernels this library has launched since the last reset (bench.py's gpu_launches) */
long long   spc_launch_count(int reset);
/* the SPC_* tuning knobs are read from the environment once per process; re-read them (dev probes only) */
void        spc_reload_env(void);

/* ---- convolution ------------------------------------------------------------------------ */
/* y = conv(pad+halo(x), w) + bias.   Replaces spatial.py:1019-1029 (ZeroPad2d :1020,
 * copy_halo_exchange_values :405-413, nn.Conv2d.forward :1027).  y: [N][K][Ho][Wo].
 * bias may be NULL.  workspace: spc_conv_workspace_bytes() bytes (may be NULL if 0). */
int spc_conv2d_fwd(const spc_conv_desc* d, const void* x, const spc_halo* halo, const void* w,
                   const void* bias, void* y, void* workspace, size_t workspace_bytes,
                   void* stream);

/* The same convolution in two stream-ordered halves, so that the halo exchange (on a second
 * stream) overlaps the bulk of the compute -- the design the reference left as dead code
 * (spatial.py:415-866 make_tensor_halo_compute / compute_halo_exchange / merge_final_image):
 *   interior: the whole tile with ZERO padding (no halo needed; tcgen05 where the shape qualifies);
 *   boundary: recompute the output rows/cols whose window reaches a received strip. */
int spc_conv2d_fwd_interior(const spc_conv_desc* d, const void* x, const void* w, const void* bias,
                            void* y, void* workspace, size_t workspace_bytes, void* stream);
int spc_conv2d_fwd_boundary(const spc_conv_desc* d, const void* x, const spc_halo* halo,
                            const void* w, const void* bias, void* y, void* stream);

/* dx = crop(dgrad(dy, w)) -- autograd of spatial.py:1027 followed by ZeroPad2d backward.
 * Reference semantics (SURVEY 8a N2): received halos are constants, so no gradient is sent
 * back to neighbours; dx gets only this tile's own dy contributions.  dx: [N][C][H][W]. */
int spc_conv2d_dgrad(const spc_conv_desc* d, const void* dy, const void* w, void* dx,
                     void* workspace, size_t workspace_bytes, void* stream);

/* dw[K][C][R][S] (fp32) and db[K] (fp32, may be NULL) over the padded tile INCLUDING the
 * received halos (autograd of spatial.py:1027 w.r.t. weight/bias).  accumulate != 0 adds
 * into dw/db instead of overwriting. */
int spc_conv2d_wgrad(const spc_conv_desc* d, const void* x, const spc_halo* halo, const void* dy,
                     float* dw, float* db, int accumulate, void* workspace,
                     size_t workspace_bytes, void* stream);

size_t spc_conv_workspace_bytes(const spc_conv_desc* d, int op /*0 fwd, 1 dgrad, 2 wgrad*/);
/* 1 if the tcgen05 (tensor-core) kernel will be used for this op, else 0 (direct kernel) */
int    spc_conv_uses_tcgen05(const spc_conv_desc* d, int op);
/* output extent of a tile: Ho = (H + 2*pad_h - R)/stride_h + 1 */
void   spc_conv_out_shape(const spc_conv_desc* d, int* Ho, int* Wo);

/* ---- pooling ---------------------------------------------------------------------------- */
/* Replaces Pool.forward (spatial.py:1503-1509): halo_exchange_layer + nn.{Max,Avg}Pool2d with
 * padding=0 on the explicitly zero-padded tile (so avg always divides by k*k and max sees 0 at
 * true image borders). */
int spc_pool2d_fwd(const spc_pool_desc* d, const void* x, const spc_halo* halo, void* y, void* stream);
/* dx = crop(pool backward); max routes to the first maximal element (ATen semantics). */
int spc_pool2d_bwd(const spc_pool_desc* d, const void* x, const spc_halo* halo, const void* dy,
                   void* dx, void* stream);

/* ---- fused BatchNorm2d (training mode, per-tile statistics) + ReLU ------------------------ *
 * The cells of the spatial stages chain ReLU -> conv -> nn.BatchNorm2d (models/amoebanet.py:365-398 of the
 * reference) / BatchNorm2d -> ReLU -> conv (resnet_spatial.py:165-180) as separate eager kernels; statistics
 * are over the LOCAL tile only (SURVEY 8a N4).  These four entry points do normalisation + the following ReLU
 * in one HBM pass each way.  y, z, dz, dy: [N][C][H*W] (NCHW, H*W % 8 == 0), dtype SPC_F32 | SPC_BF16;
 * all per-channel vectors are fp32 device arrays of C elements.
 *   spc_bn_stats     : sum[c] = sum y, sumsq[c] = sum y^2                          (replaces the statistics pass)
 *   spc_bn_apply     : z = relu?((y - mean[c]) * rstd[c] * gamma[c] + beta[c])     (BN apply + nn.ReLU)
 *   spc_bn_bwd_reduce: dsum[c] = sum g, dsumx[c] = sum g * xhat, g = dz * [z > 0]  (= dbeta, dgamma)
 *   spc_bn_bwd_apply : dy = gamma * rstd * (g - dsum/M - xhat * dsumx/M), M = N*H*W */
int spc_bn_stats(int N, int C, long long HW, int dtype, const void* y, float* sum, float* sumsq, void* stream);
int spc_bn_apply(int N, int C, long long HW, int dtype, const void* y, const float* mean, const float* rstd,
                 const float* gamma, const float* beta, int relu, void* z, void* stream);
int spc_bn_bwd_reduce(int N, int C, long long HW, int dtype, const void* dz, const void* y, const float* mean,
                      const float* rstd, const float* gamma, const float* beta, int relu, float* dsum,
                      float* dsumx, void* stream);
int spc_bn_bwd_apply(int N, int C, long long HW, int dtype, const void* dz, const void* y, const float* mean,
                     const float* rstd, const float* gamma, const float* beta, int relu, const float* dsum,
                     const float* dsumx, void* dy, void* stream);

/* ---- halo strips ------------------------------------------------------------------------ */
/* Pack the strips a tile SENDS (spatial.py:336-357: the first/last halo rows/cols inside the
 * tile, .clone()d per direction) into send[d] for every d with send[d] != NULL.  send[d] may be
 * a peer-GPU pointer (CUDA IPC mapping): one kernel writes all strips straight into the
 * neighbours' receive buffers over NVLink. Strip d goes to the neighbour in direction d, who
 * receives it as ITS strip 8-d (tags, spatial.py:170-172). */
int spc_halo_pack(int N, int C, int H, int W, int halo_h, int halo_w, int dtype, const void* x,
                  void* const send[9], void* stream);
/* Materialise the padded tile (halo_exchange_layer.forward output, spatial.py:1404-1413):
 * y[N][C][H+2hh][W+2hw] = x in the middle, strips / zeros around. */
int spc_halo_pad(int N, int C, int H, int W, int halo_h, int halo_w, int dtype, const void* x,
                 const spc_halo* halo, void* y, void* stream);
/* Backward of spc_halo_pad: crop the middle. */
int spc_halo_crop(int N, int C, int H, int W, int halo_h, int halo_w, int dtype, const void* dy,
                  void* dx, void* stream);

/* ---- peer-memory halo transport (one process per GPU, NVLink / NVSwitch) ------------------
 * Replaces dist.isend/irecv + torch.cuda.synchronize() fences (spatial.py:351-393,401-403).
 * A "mailbox" is a device allocation owned by this rank holding `slots` receive areas of
 * `bytes` each plus per-slot arrival flags.  Peers map it with CUDA IPC and their pack kernel
 * (spc_halo_pack with peer pointers) writes into it; ordering uses device-side flags
 * (release/acquire at system scope), never a host synchronisation. */
typedef struct spc_mailbox spc_mailbox;
#define SPC_IPC_HANDLE_BYTES 64
int   spc_mailbox_create(spc_mailbox** out, size_t bytes, int nflags);
void  spc_mailbox_destroy(spc_mailbox* mb);
void* spc_mailbox_data(spc_mailbox* mb);                       /* local device pointer */
int   spc_mailbox_export(spc_mailbox* mb, unsigned char handle[SPC_IPC_HANDLE_BYTES]);
/* Map a peer's mailbox (handle obtained from the peer through torch.distributed). */
int   spc_mailbox_open(spc_mailbox** out, const unsigned char handle[SPC_IPC_HANDLE_BYTES],
                       size_t bytes, int nflags);
/* Fused protocol steps (one kernel each).  post: wait until local ack flags ack_idx[d] reach
 * ack_seq (0 = do not wait) -> pack every strip d with send[d] != NULL into send[d] (peer slot) ->
 * when the whole grid is done, publish `seq` on peers[d]'s arrival flag arrival_idx[d].
 * collect: wait for local arrival flags arrival_idx[d] >= seq -> copy bytes[d] from src[d] (local
 * mailbox slot) to dst[d] -> publish `seq` on peers[d]'s ack flag ack_idx[d]. */
int spc_halo_post(int N, int C, int H, int W, int halo_h, int halo_w, int dtype, const void* x,
                  void* const send[9], spc_mailbox* self, spc_mailbox* const peers[9],
                  const int ack_idx[9], uint32_t ack_seq, const int arrival_idx[9], uint32_t seq,
                  void* stream);
int spc_halo_collect(void* const dst[9], const void* const src[9], const size_t bytes[9],
                     spc_mailbox* self, spc_mailbox* const peers[9], const int arrival_idx[9],
                     uint32_t seq, const int ack_idx[9], void* stream);
/* Graph-capturable variants (what torchgems.halo_transport.PeerTransport uses): no host-side state in the
 * launch arguments.  The sequence number s of the exchange is (local flag seq_idx) + 1, read on the device;
 * its parity selects the half of the double-buffered slot (send0[d] / src0[d] + (s&1)*slot_bytes) and the
 * flag bank (index + (s&1)*9).  post waits for the acks of sequence s-2 (s <= 2: none); collect waits for
 * the arrivals of s, copies out, acks, and its last block stores s to flag seq_idx.  post and collect of one
 * exchange must be enqueued in that order on one stream.  counter_idx: a flag word private to the layer's
 * slot, used as the grid-completion counter (exchanges of different layers may run on different streams).
 * The flag waits are bounded: after SPCONV_SPIN_TIMEOUT_S seconds (default 120, 0 = unbounded) the kernel
 * prints the direction it is stuck on and traps, so a dead peer surfaces as a CUDA error, not a hang.
 * Replaces the same reference lines as spc_halo_post / spc_halo_collect (spatial.py:336-403). */
int spc_halo_post_auto(int N, int C, int H, int W, int halo_h, int halo_w, int dtype, const void* x,
                       void* const send0[9], size_t slot_bytes, spc_mailbox* self,
                       spc_mailbox* const peers[9], const int ack_idx0[9], const int arrival_idx0[9],
                       int seq_idx, int counter_idx, void* stream);
int spc_halo_collect_auto(void* const dst[9], const void* const src0[9], const size_t bytes[9],
                          size_t slot_bytes, spc_mailbox* self, spc_mailbox* const peers[9],
                          const int arrival_idx0[9], const int ack_idx0[9], int seq_idx, int counter_idx,
                          void* stream);
/* After writes to peer `mb` enqueued on `stream`: publish sequence number `seq` on flag `idx`. */
int   spc_mailbox_signal(spc_mailbox* peer_mb, int idx, uint32_t seq, void* stream);
/* Make `stream` wait (on device) until local flag `idx` reaches `seq`. */
int   spc_mailbox_wait(spc_mailbox* mb, int idx, uint32_t seq, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SPCONV_H_ */
