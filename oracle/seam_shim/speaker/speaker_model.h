// TEST INFRASTRUCTURE ONLY: stand-in for the C++ runtime's model interface (runtime/core/speaker/speaker_model.h of
// WeSpeaker), declared from its public signature so that wespeaker::B200SpeakerModel (csrc/runtime) compiles and is
// tested without the WeSpeaker runtime tree.  Only the virtual the B200 back-end overrides is declared.  Building against
// this stand-in does not check compatibility with the real header; the oracle/_ref/libb200_seam.so build does, where the
// WeSpeaker sources are present.
#ifndef SPEAKER_SPEAKER_MODEL_H_
#define SPEAKER_SPEAKER_MODEL_H_

#include <vector>

namespace wespeaker {

class SpeakerModel {
 public:
  virtual ~SpeakerModel() = default;
  virtual void ExtractEmbedding(const std::vector<std::vector<float>>& feats, std::vector<float>* embed) = 0;
};

}  // namespace wespeaker

#endif  // SPEAKER_SPEAKER_MODEL_H_
