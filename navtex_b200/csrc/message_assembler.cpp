#include "message_assembler.h"

#include "demod.cuh"

namespace nvx {

namespace {
constexpr size_t kTextCap = 4999;   // the reference's buffers are char[5000] (nav_b_sm.h:97-98)
void bounded_append(std::string& dst, const std::string& src) {
    if (dst.size() >= kTextCap) return;
    dst.append(src, 0, kTextCap - dst.size());
}
}  // namespace

MessageAssembler::MessageAssembler() {
    // the two patterns of message_line_out (nav_b_sm.C:69, :80); POSIX ERE, as there
    regcomp(&som_, "(CZC|Z.ZC|ZC.C|ZCZ.) +([A-Z][A-Z])([0-9][0-9])", REG_EXTENDED);
    regcomp(&eom_, "NNN.*|N.NN.*|NN.N.*", REG_EXTENDED);
}
MessageAssembler::~MessageAssembler() {
    regfree(&som_);
    regfree(&eom_);
}

void MessageAssembler::resize(int channels) { ch_.assign((size_t)channels, Channel()); }
void MessageAssembler::reset() { ch_.assign(ch_.size(), Channel()); }
void MessageAssembler::reset_channel(int ch) { ch_[(size_t)ch] = Channel(); }

namespace {
// Necessary conditions of the two patterns, checked before paying for regexec (most lines are plain text):
// every start-of-message alternative contains three of {Z, C} and is followed by a blank and two digits;
// every end-of-message alternative contains three N.
void line_census(const std::string& line, int* zc, int* n, bool* blank, bool* digit) {
    *zc = *n = 0;
    *blank = *digit = false;
    for (char ch : line) {
        if (ch == 'Z' || ch == 'C') ++*zc;
        else if (ch == 'N') ++*n;
        else if (ch == ' ') *blank = true;
        else if (ch >= '0' && ch <= '9') *digit = true;
    }
}
}  // namespace

// message_line_out, nav_b_sm.C:56-97
void MessageAssembler::line_done(Channel& c, int stream, int freq, std::vector<AssembledMessage>* out) {
    regmatch_t m[4];
    if (c.in_message) {
        bounded_append(c.text, c.line);
        bounded_append(c.text, "\n");
    }
    int zc, nn;
    bool blank, digit;
    line_census(c.line, &zc, &nn, &blank, &digit);
    if (zc >= 3 && blank && digit && regexec(&som_, c.line.c_str(), 4, m, 0) == 0) {
        c.text.clear();
        bounded_append(c.text, c.line);
        bounded_append(c.text, "\n");
        // B1B2 and B3B4 are appended to whatever bbbb already holds and the result is cut at four
        // characters (strncat + [4] = 0, nav_b_sm.C:74-76): a second ZCZC before NNNN keeps the old id
        c.bbbb.append(c.line, (size_t)m[2].rm_so, (size_t)(m[2].rm_eo - m[2].rm_so));
        c.bbbb.append(c.line, (size_t)m[3].rm_so, (size_t)(m[3].rm_eo - m[3].rm_so));
        if (c.bbbb.size() > 4) c.bbbb.resize(4);
        c.in_message = true;
    } else if (nn >= 3 && regexec(&eom_, c.line.c_str(), 1, m, 0) == 0) {
        if (c.in_message) out->push_back(AssembledMessage{stream, freq, c.bbbb, c.text});
        c.text.clear();
        c.bbbb.clear();
        c.in_message = false;
    }
    c.line.clear();
}

void MessageAssembler::feed(int ch, int stream, int freq, const unsigned char* ev, size_t n,
                            std::vector<AssembledMessage>* out) {
    Channel& c = ch_[(size_t)ch];
    for (size_t k = 0; k < n; ++k) {
        const unsigned char b = ev[k];
        if (b == '\n') {
            line_done(c, stream, freq, out);
        } else if (b == kEvAbort) {
            // message_abort, nav_b_sm.C:44-52: a message in progress is stored as it stands, then init()
            if (c.in_message) out->push_back(AssembledMessage{stream, freq, c.bbbb, c.text});
            c = Channel();
        } else if (c.line.size() < kTextCap) {
            c.line.push_back((char)b);
        }
    }
}

}  // namespace nvx
