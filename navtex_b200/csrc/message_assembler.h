// message_assembler.h -- host half of byte_state_machine: line buffer, ZCZC / NNNN framing,
// B1B2B3B4 extraction and the add_message hand-off (receiver/nav_b_sm.C:44-52, :56-97), driven by
// the character / line / abort event stream the demod kernel emits per channel.
#pragma once
#include <regex.h>

#include <string>
#include <vector>

namespace nvx {

struct AssembledMessage {
    int stream, freq;
    std::string bbbb, text;
};

class MessageAssembler {
  public:
    MessageAssembler();
    ~MessageAssembler();
    MessageAssembler(const MessageAssembler&) = delete;
    MessageAssembler& operator=(const MessageAssembler&) = delete;

    void resize(int channels);
    void reset();
    // drop channel ch's partial line and message without delivering them (nvx_engine_reset_streams)
    void reset_channel(int ch);
    // feed `n` event bytes of channel `ch`; completed messages are appended to `out`
    void feed(int ch, int stream, int freq, const unsigned char* ev, size_t n, std::vector<AssembledMessage>* out);

    // a channel's partial line and message (nvx_engine_save_streams / nvx_engine_load_streams)
    struct Channel {
        std::string line, text, bbbb;
        bool in_message = false;
    };
    const Channel& channel(int ch) const { return ch_[(size_t)ch]; }
    void set_channel(int ch, const Channel& c) { ch_[(size_t)ch] = c; }

  private:
    void line_done(Channel& c, int stream, int freq, std::vector<AssembledMessage>* out);
    std::vector<Channel> ch_;
    regex_t som_, eom_;
};

}  // namespace nvx
