// rpsf_ops.h — type-erased launch table, one instance per patch size P.
// Each size is compiled in its own translation unit (rpsf_inst.cu with -DRPSF_P=...).
#pragma once
#include <cuda_runtime.h>
#include "rpsf_kernels.cuh"
#include "rpsf_stream.cuh"

namespace rpsf {

enum DType : int { DT_F32 = 0, DT_F64 = 1 };

struct Ops {
  int P;
  // set shared-memory attributes for the current device; returns a cudaError_t
  int (*init)();
  // the row passes write the band buffer `bands` (rpsf_bands.cuh)
  int (*k1)(int dt, const void* image, void* bands, const RowBands& rb, const void* tw, const void* win,
            const ApplyGeom& g, int batch, cudaStream_t s);
  // persistent bulk-async K1 (rpsf_stream.cuh); `bulk_ok`: frame base, pitch and frame stride are 16-byte aligned
  int (*k1s)(int dt, const void* image, void* bands, const RowBands& rb, const void* tw, const void* win,
             const ApplyGeom& g, int batch, int bulk_ok, int sm_count, cudaStream_t s);
  // the column pass reads the band buffer and writes the spectrum workspace `spec`
  int (*k2)(int dt, const void* bands, const RowBands& rb, void* spec, const void* kmain, const void* knyq,
            const int* active, const void* tw, const void* win, const ApplyGeom& g, int batch, int sm_count,
            cudaStream_t s);
  // the column pass of a transform stack (k2_stack): n_kernels kernels at kmain + m * kmain_stride / knyq + m *
  // knyq_stride, spectra of kernel m at spec + m * kspec_stride (complex elements); k2s_ok(dt): it exists for this
  // patch size and dtype (the pipelined stage ring fits)
  int (*k2s)(int dt, const void* bands, const RowBands& rb, void* spec, long long kspec_stride, const void* kmain,
             long long kmain_stride, const void* knyq, long long knyq_stride, int n_kernels, const int* active,
             const void* tw, const void* win, const ApplyGeom& g, int batch, int sm_count, cudaStream_t s);
  int (*k2s_ok)(int dt);
  int (*k3)(int dt, const void* spec, void* out, const int2* corners, const int* items, int n_items,
            const void* tw, const void* win, int store_only, const ApplyGeom& g, int batch, cudaStream_t s);
  // single-launch overlap-add: `teams` teams per CTA, `seg_w` output columns per CTA
  int (*k3g)(int dt, const void* spec, void* out, const RowTile* tiles, int n_tiles, const RowGroup* groups,
             const int* items, const void* tw, const void* win, int teams, int seg_w, const ApplyGeom& g,
             int batch, cudaStream_t s);
  // persistent bulk-async K3 (rpsf_stream.cuh): chains of half-overlapping groups walked in registers
  // `mirrors` (may be null): peer buffers that receive every store too (OutMirrors, rpsf_stream.cuh)
  int (*k3s)(int dt, const void* spec, void* out, const StreamTask* tasks, const unsigned* codes, int n_warp_items,
             const void* tw, const void* win, const ApplyGeom& g, int batch, int sm_count, const OutMirrors* mirrors,
             cudaStream_t s);
  // teams per warp of the streaming kernels (tasks are laid out in groups of this many)
  int (*stream_tpw)();
  // shared memory the gather kernel needs for that shape (bytes), to size `teams`
  size_t (*k3g_smem)(int dt, int teams, int seg_w);
  int (*prep)(int dt, int kernel_dt, const void* full, void* kmain, void* knyq, int n_patches, cudaStream_t s);
  int (*fft2)(int dt, int in_dt, const void* values, void* out, const void* tw, long long n_patches,
              cudaStream_t s);
  // gradient with respect to the transfer kernel (rpsf_kgrad.cuh): conj(X) G / P^2 summed over `batch` frames of the
  // forward (xspec) and adjoint (gspec) band buffers, into the (n, P, P) cube `out` at slots active[a]
  int (*kgrad)(int dt, const void* xspec, const RowBands& xb, const void* gspec, const RowBands& gb, void* out,
               const int* active, const void* tw, const void* win, int n_active, int batch, cudaStream_t s);
  // adjoint of fft2 (rpsf_construct_grad.cuh): out (n, P, P) real = Re(fft2(conj(grad))), through the complex
  // (n, P, P) cube `scratch`
  int (*fft2_adjoint)(int dt, const void* grad, void* scratch, void* out, const void* tw, long long n_patches,
                      cudaStream_t s);
};

const Ops* ops_for(int P);   // nullptr when P is unsupported

const Ops* ops_p16();
const Ops* ops_p32();
const Ops* ops_p64();
const Ops* ops_p128();
const Ops* ops_p256();
const Ops* ops_p512();

}  // namespace rpsf
