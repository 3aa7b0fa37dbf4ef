// kb_step_kernel.cuh -- the lane-group step kernel's body, its block sizes and launch bounds.  Included by kb_b200.cu,
// which instantiates it on the runtime Layout (kb_step_kernel<LPE>), and by the source kb_create compiles at run time
// for one batch's layout (kb_jit.h), which instantiates it on a compile-time layout.
#pragma once
#include "kb_toi.cuh"

namespace kb {

// threads per block.  The warps of a block rendezvous at the phase boundaries (KB_T in kb_step.cuh) and so share
// instruction-cache lines: with one warp per block the 4-lane kernel spent 10 of 17 cycles per issue waiting for
// instructions (profiles/ncu_step_kernel_r01_c5_block32_before.txt).  Measured on C5 (2^18 envs, kilobot-steps/s):
// 32 threads 70 M, 64 threads 114 M, 96 threads 132 M, 128 threads 139 M, 192 threads 132 M; the wider kernels are best
// at two warps (C2: 64 threads 1.215 ms, 128 threads 1.239 ms; C3: 5.39 vs 5.55 ms).
#ifndef KB_BLOCK4
#define KB_BLOCK4 128
#endif
#ifndef KB_BLOCK8
#define KB_BLOCK8 64
#endif
#ifndef KB_BLOCK16
#define KB_BLOCK16 64
#endif
#ifndef KB_MINBLOCKS16
#define KB_MINBLOCKS16 6
#endif
#ifndef KB_MINBLOCKS8
#define KB_MINBLOCKS8 3
#endif
#ifndef KB_MINBLOCKS4
#define KB_MINBLOCKS4 6   /* 6 blocks of 64 threads per SM: <= 168 registers (C5: 96 resident envs per SM) */
#endif
#ifndef KB_BLOCK32
#define KB_BLOCK32 64
#endif
#define KB_BLOCK_OF(LPE) ((LPE) == 4 ? KB_BLOCK4 : ((LPE) == 8 ? KB_BLOCK8 : ((LPE) == 16 ? KB_BLOCK16 : KB_BLOCK32)))
// __launch_bounds__ of the step kernel
#define KB_STEP_BOUNDS(LPE) KB_BLOCK_OF(LPE), (LPE == 32 ? (512 / KB_BLOCK32) : (KB_BLOCK_OF(LPE) > 64 ? (384 / KB_BLOCK_OF(LPE)) : (LPE == 16 ? KB_MINBLOCKS16 : (LPE == 4 ? KB_MINBLOCKS4 : KB_MINBLOCKS8))))

// The batch is padded to a whole number of blocks (numEnvs <= grid * EPB): every lane of the step kernel owns
// a real environment, so the groups of a warp can run in lock step.  Padding envs replicate the inputs of the
// last real env and never write outputs.  Everything the layout covers is read through s.L, so that a compile-time
// layout turns offsets, counts and constants into immediates.
template <int LPE, class LT>
__device__ __forceinline__ void stepKernelBody(const KernelArgs& a, const LT& layout) {
  constexpr int EPB = KB_BLOCK_OF(LPE) / LPE;
  const int slot = threadIdx.x / LPE;
  const int env = a.envOffset + blockIdx.x * EPB + slot;
  const int envIn = min(env, a.numEnvs - 1);
  Sim<LPE, true, LT> s(layout);
  s.g.init();
  s.bind(slot);
  s.blob = a.blobs + (size_t)env * s.L.blobWords;
  const int scene = a.envScene ? (int)reinterpret_cast<const uint32_t*>(s.blob)[s.L.oHdr + H_SCENE] : 0;   // (last reset's)
  s.px = a.proxies + (size_t)scene * s.L.Pp;
  s.bc = a.bodies + (size_t)scene * s.L.Bp;
  s.lights = a.lights + (size_t)scene * (s.L.numLights > 0 ? s.L.numLights : 1);
  s.S = s.L.B;
#ifdef KB_PROFILE
  s.profOut = a.prof ? a.prof + (size_t)envIn * KB_PROF_SLOTS : nullptr;
  if (s.profOut && s.g.lane == 0) s.profOut[13] = s.profOut[14] = s.profOut[15] = 0ull;
#endif
  s.loadState();
  s.initScratch();
  const int A = a.actionMode == KB_ACTION_KILOBOTS ? 2 * s.L.N : s.L.A;
  const double* act = a.action ? a.action + (size_t)envIn * A : nullptr;
  // the doubled warp barriers after setKilobotActions and senseControl are redundant but kept: without them the
  // compiler schedules this kernel differently (measured in SASS)
  if (a.actionMode == KB_ACTION_KILOBOTS) {
    setKilobotActions(s, act, s.g.lane, LPE);
    s.g.usync();
  }
  s.g.usync();
  if (a.task.mode != KB_TASK_CONST && s.g.lane == 0 && env < a.numEnvs)  // task layer, include/kb_b200.h
    taskBegin(s, a, env);
  for (int step = 0; step < s.L.stepsPerAction; ++step) {
    __syncthreads();  // keeps the warps of a block in the same phase (see KB_T in kb_step.cuh)
    if (a.actionMode == KB_ACTION_LIGHT && act && s.L.numLights > 0) {
      if (s.g.lane == 0) lightStep(s, act);
      s.g.usync();
    }
    senseControl(s, s.g.lane, LPE);
    s.g.usync();
    s.g.usync();
    s.worldStep();
  }
  if (env < a.numEnvs) s.gather(a, env);
  s.storeState();
#ifdef KB_PROFILE
  s.tp[12] += clock64() - s.tlast;
  if (a.prof && s.g.lane == 0 && env < a.numEnvs)
    for (int i = 0; i < 13; ++i) a.prof[(size_t)env * KB_PROF_SLOTS + i] = (unsigned long long)s.tp[i];
#endif
}

}  // namespace kb
