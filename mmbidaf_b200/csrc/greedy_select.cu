// Greedy sentence selection on the device (decode.greedy_search, reference evaluate.py:185-202): from the per-step arg-max of a
// summary roll-out (B, S) and the text lengths, the chosen sentence indices of every video, so that only those (and not the (B, S, M)
// distributions) go to the host.  The rule, per video in step order: the EOS row `len - 1` ends the summary; an index past it names
// no sentence of the transcript and is skipped (evaluate.py:195, :255-256); anything else is kept, repeats included.
#include "common.cuh"

namespace mmb {
namespace {

__global__ void __launch_bounds__(128) greedy_select_kernel(const long long* __restrict__ argmax, const int32_t* __restrict__ len,
                                                            int32_t* __restrict__ sel, int32_t* __restrict__ count, int B, int S) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const long long eos = (long long)len[b] - 1;
  const long long* am = argmax + (size_t)b * S;
  int32_t* out = sel + (size_t)b * S;
  int c = 0;
  for (int s = 0; s < S; ++s) {
    const long long k = am[s];
    if (k == eos) break;
    if (k > eos) continue;
    out[c++] = (int32_t)k;
  }
  count[b] = c;
  for (int s = c; s < S; ++s) out[s] = -1;
}

}  // namespace
}  // namespace mmb

extern "C" int mmb_greedy_select(const long long* argmax, const int32_t* text_len, int32_t* sel, int32_t* count, int B, int S,
                                 mmb_stream_t stream) {
  MMB_REQUIRE(argmax && text_len && sel && count && B > 0 && S > 0, MMB_ERR_INVALID, "mmb_greedy_select: B=%d S=%d", B, S);
  mmb::greedy_select_kernel<<<(B + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(argmax, text_len, sel, count, B, S);
  return mmb::check_launch("greedy_select_kernel");
}
