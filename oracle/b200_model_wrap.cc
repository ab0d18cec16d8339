// TEST INFRASTRUCTURE ONLY: C entry point over wespeaker::B200SpeakerModel (wespeaker_b200/csrc/runtime), reached the
// way the C++ runtime's SpeakerEngine reaches its model: through a SpeakerModel pointer, one chunk of [T][F] feature rows
// per virtual ExtractEmbedding call.  The chunking, mean normalisation and averaging around it are done by the caller
// (tests/test_speaker_engine.py, with oracle/speaker_engine_py.py pinned on the runtime's own outputs).
#include <cstring>
#include <memory>
#include <vector>

#include "b200_speaker_model.h"

extern "C" int b200_model_extract_chunks(const char* flat_model_path, int device, const float* feats, int nchunks, int T,
                                         int F, float* emb_out, int emb_size) {
    auto b200 = std::make_unique<wespeaker::B200SpeakerModel>(flat_model_path, device);
    if (b200->EmbeddingSize() != emb_size) return -1;
    wespeaker::SpeakerModel* model = b200.get();
    std::vector<std::vector<float>> chunk(T, std::vector<float>(F));
    std::vector<float> emb;
    for (int c = 0; c < nchunks; ++c) {
        for (int t = 0; t < T; ++t)
            std::memcpy(chunk[t].data(), feats + ((size_t)c * T + t) * F, sizeof(float) * F);
        model->ExtractEmbedding(chunk, &emb);
        if ((int)emb.size() != emb_size) return -2;
        std::memcpy(emb_out + (size_t)c * emb_size, emb.data(), sizeof(float) * emb_size);
    }
    return 0;
}
