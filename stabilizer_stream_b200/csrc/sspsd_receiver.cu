// sspsd_receiver.cu -- UDP ingest for the frame path: recvmmsg into a pinned slot ring, handed to the
// batched decoder (K1) as one strided frame array.
//
// Replaces the per-datagram loop of the reference (src/source.rs:81-93 socket set-up, 159-165
// `socket.read(&mut buf)` -> Frame::from_bytes -> loss.update -> traces per packet): datagrams are
// collected many at a time, stay in page-locked memory, and cross PCIe once per batch.
#include <arpa/inet.h>
#include <netinet/in.h>
#include <poll.h>
#include <sys/socket.h>
#include <unistd.h>

#include <cerrno>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "sspsd_cascade.cuh"

namespace sspsd {

class Receiver {
public:
    ~Receiver()
    {
        if (fd_ >= 0) close(fd_);
        if (buf_) {
            if (pinned_)
                cudaFreeHost(buf_);
            else
                free(buf_);
        }
    }

    int init(const char* ip, uint16_t port, uint32_t slot_bytes, uint32_t n_slots, int flags)
    {
        if (!ip || slot_bytes < SSPSD_HEADER_SIZE || slot_bytes % 8 || n_slots == 0) {
            set_error("receiver: bad argument (slot_bytes must be a multiple of 8)");
            return SSPSD_EINVAL;
        }
        in_addr addr{};
        if (inet_pton(AF_INET, ip, &addr) != 1) {
            set_error("receiver: not an IPv4 address");
            return SSPSD_EINVAL;
        }
        slot_ = slot_bytes;
        n_slots_ = n_slots;
        const size_t bytes = (size_t)slot_ * n_slots_;
        if (flags & SSPSD_RECV_PAGEABLE) {
            if (posix_memalign((void**)&buf_, 4096, bytes)) return SSPSD_ENOMEM;
        } else {
            SSPSD_CUDA(cudaHostAlloc((void**)&buf_, bytes, cudaHostAllocDefault));
            pinned_ = true;
        }
        fd_ = socket(AF_INET, SOCK_DGRAM, IPPROTO_UDP);
        if (fd_ < 0) return sys_error("socket");
        // source.rs:84-86: 1 MiB receive buffer, reuse address
        int rcv = 1 << 20, one = 1;
        setsockopt(fd_, SOL_SOCKET, SO_RCVBUF, &rcv, sizeof(rcv));
        if (setsockopt(fd_, SOL_SOCKET, SO_REUSEADDR, &one, sizeof(one)) < 0) return sys_error("SO_REUSEADDR");
        // source.rs:87-89: join the group when the address is multicast
        if ((ntohl(addr.s_addr) >> 28) == 0xe) {
            ip_mreq mreq{};
            mreq.imr_multiaddr = addr;
            mreq.imr_interface.s_addr = htonl(INADDR_ANY);
            if (setsockopt(fd_, IPPROTO_IP, IP_ADD_MEMBERSHIP, &mreq, sizeof(mreq)) < 0) return sys_error("IP_ADD_MEMBERSHIP");
        }
        sockaddr_in sa{};
        sa.sin_family = AF_INET;
        sa.sin_addr = addr;  // source.rs:92-93 (non-windows): bind to the given address
        sa.sin_port = htons(port);
        if (bind(fd_, (sockaddr*)&sa, sizeof(sa)) < 0) return sys_error("bind");
        socklen_t sl = sizeof(sa);
        if (getsockname(fd_, (sockaddr*)&sa, &sl) == 0) port_ = ntohs(sa.sin_port);
        msgs_.resize(n_slots_);
        iov_.resize(n_slots_);
        len_.assign(n_slots_, 0);
        return SSPSD_OK;
    }

    uint16_t port() const { return port_; }
    size_t slot_bytes() const { return slot_; }
    uint64_t datagrams() const { return total_; }

    // Next run of equally sized datagrams: frames = first slot, stride = slot_bytes().  The run stays
    // valid until the next call.  n_frames == 0 after timeout_ms without traffic (source.rs:83 uses 1 s).
    int recv(uint32_t max_frames, int timeout_ms, const uint8_t** frames, size_t* n_frames, size_t* frame_len)
    {
        *frames = nullptr;
        *n_frames = 0;
        *frame_len = 0;
        if (max_frames == 0) return SSPSD_OK;
        if (head_ == tail_) {
            head_ = tail_ = 0;
            pollfd pfd{fd_, POLLIN, 0};
            int pr;
            do {
                pr = poll(&pfd, 1, timeout_ms);
            } while (pr < 0 && errno == EINTR);
            if (pr < 0) return sys_error("poll");
            if (pr == 0) return SSPSD_OK;
            const uint32_t want = max_frames < n_slots_ ? max_frames : n_slots_;
            for (uint32_t i = 0; i < want; ++i) {
                iov_[i].iov_base = buf_ + (size_t)i * slot_;
                iov_[i].iov_len = slot_;
                std::memset(&msgs_[i], 0, sizeof(mmsghdr));
                msgs_[i].msg_hdr.msg_iov = &iov_[i];
                msgs_[i].msg_hdr.msg_iovlen = 1;
            }
            int got;
            do {
                got = recvmmsg(fd_, msgs_.data(), want, MSG_DONTWAIT, nullptr);
            } while (got < 0 && errno == EINTR);
            if (got < 0) {
                if (errno == EAGAIN || errno == EWOULDBLOCK) return SSPSD_OK;
                return sys_error("recvmmsg");
            }
            for (int i = 0; i < got; ++i) {
                // a datagram longer than the slot is cut by the kernel, exactly like the reference's
                // 2048-byte read buffer (source.rs:160); the payload-size check of the decoder reports it
                len_[i] = msgs_[i].msg_len;
            }
            tail_ = (uint32_t)got;
            total_ += (uint64_t)got;
        }
        // longest run of equal lengths from head_, at most max_frames
        const uint32_t l = len_[head_];
        uint32_t e = head_ + 1;
        while (e < tail_ && e - head_ < max_frames && len_[e] == l) ++e;
        *frames = buf_ + (size_t)head_ * slot_;
        *n_frames = e - head_;
        *frame_len = l;
        head_ = e;
        return SSPSD_OK;
    }

private:
    int sys_error(const char* what)
    {
        set_error(std::string("receiver: ") + what + ": " + std::strerror(errno));
        return SSPSD_EIO;
    }
    int fd_ = -1;
    uint16_t port_ = 0;
    uint8_t* buf_ = nullptr;
    bool pinned_ = false;
    size_t slot_ = 0;
    uint32_t n_slots_ = 0, head_ = 0, tail_ = 0;
    uint64_t total_ = 0;
    std::vector<mmsghdr> msgs_;
    std::vector<iovec> iov_;
    std::vector<uint32_t> len_;
};

}  // namespace sspsd

using namespace sspsd;

struct sspsd_receiver {
    Receiver r;
};

extern "C" {

int32_t sspsd_receiver_create(const char* ip, uint16_t port, uint32_t slot_bytes, uint32_t n_slots, int32_t flags,
                              sspsd_receiver** out)
{
    if (!out) return SSPSD_EINVAL;
    *out = nullptr;
    sspsd_receiver* h = new (std::nothrow) sspsd_receiver;
    if (!h) return SSPSD_ENOMEM;
    int rc = h->r.init(ip, port, slot_bytes ? slot_bytes : 2048, n_slots ? n_slots : 1024, flags);
    if (rc) {
        delete h;
        return rc;
    }
    *out = h;
    return SSPSD_OK;
}

void sspsd_receiver_destroy(sspsd_receiver* h) { delete h; }

int32_t sspsd_receiver_info(const sspsd_receiver* h, uint16_t* port, size_t* slot_bytes, uint64_t* datagrams)
{
    if (!h) return SSPSD_EINVAL;
    if (port) *port = h->r.port();
    if (slot_bytes) *slot_bytes = h->r.slot_bytes();
    if (datagrams) *datagrams = h->r.datagrams();
    return SSPSD_OK;
}

int32_t sspsd_receiver_recv(sspsd_receiver* h, uint32_t max_frames, int32_t timeout_ms, const uint8_t** frames,
                            size_t* n_frames, size_t* frame_len)
{
    if (!h || !frames || !n_frames || !frame_len) return SSPSD_EINVAL;
    return h->r.recv(max_frames, timeout_ms, frames, n_frames, frame_len);
}

int32_t sspsd_receiver_pump(sspsd_receiver* h, sspsd_decoder* d, sspsd_cascade* const* cascades, uint32_t n_cascades,
                            uint32_t max_frames, int32_t timeout_ms, sspsd_loss* loss, sspsd_decode_info* info)
{
    if (!h || !d) return SSPSD_EINVAL;
    if (info) std::memset(info, 0, sizeof(*info));
    const uint8_t* frames = nullptr;
    size_t n = 0, len = 0;
    int rc = h->r.recv(max_frames, timeout_ms, &frames, &n, &len);
    if (rc || n == 0) return rc;
    return sspsd_cascade_process_frames(d, cascades, n_cascades, frames, n, len, h->r.slot_bytes(), SSPSD_MEM_HOST, loss,
                                        info);
}

// The handles and the trace map are checked (an empty batch) before a run is taken from the ring, so that a bad
// argument drops no datagram.
int32_t sspsd_receiver_pump_csm(sspsd_receiver* h, sspsd_decoder* d, sspsd_csm* m, const uint32_t* traces,
                                uint32_t max_frames, int32_t timeout_ms, sspsd_loss* loss, sspsd_decode_info* info)
{
    if (!h) return SSPSD_EINVAL;
    if (info) std::memset(info, 0, sizeof(*info));
    int rc = sspsd_csm_process_frames(d, m, traces, nullptr, 0, 0, 0, SSPSD_MEM_HOST, nullptr, nullptr);
    if (rc) return rc;
    const uint8_t* frames = nullptr;
    size_t n = 0, len = 0;
    rc = h->r.recv(max_frames, timeout_ms, &frames, &n, &len);
    if (rc || n == 0) return rc;
    return sspsd_csm_process_frames(d, m, traces, frames, n, len, h->r.slot_bytes(), SSPSD_MEM_HOST, loss, info);
}

int32_t sspsd_receiver_pump_csd(sspsd_receiver* h, sspsd_decoder* d, sspsd_csd* c, uint32_t trace_x, uint32_t trace_y,
                                uint32_t max_frames, int32_t timeout_ms, sspsd_loss* loss, sspsd_decode_info* info)
{
    if (!h) return SSPSD_EINVAL;
    if (info) std::memset(info, 0, sizeof(*info));
    int rc = sspsd_csd_process_frames(d, c, trace_x, trace_y, nullptr, 0, 0, 0, SSPSD_MEM_HOST, nullptr, nullptr);
    if (rc) return rc;
    const uint8_t* frames = nullptr;
    size_t n = 0, len = 0;
    rc = h->r.recv(max_frames, timeout_ms, &frames, &n, &len);
    if (rc || n == 0) return rc;
    return sspsd_csd_process_frames(d, c, trace_x, trace_y, frames, n, len, h->r.slot_bytes(), SSPSD_MEM_HOST, loss,
                                    info);
}

int32_t sspsd_receiver_pump_zoom(sspsd_receiver* h, sspsd_decoder* d, sspsd_zoom* z, const uint32_t* traces,
                                 uint32_t max_frames, int32_t timeout_ms, sspsd_loss* loss, sspsd_decode_info* info)
{
    if (!h) return SSPSD_EINVAL;
    if (info) std::memset(info, 0, sizeof(*info));
    int rc = sspsd_zoom_process_frames(d, z, traces, nullptr, 0, 0, 0, SSPSD_MEM_HOST, nullptr, nullptr);
    if (rc) return rc;
    const uint8_t* frames = nullptr;
    size_t n = 0, len = 0;
    rc = h->r.recv(max_frames, timeout_ms, &frames, &n, &len);
    if (rc || n == 0) return rc;
    return sspsd_zoom_process_frames(d, z, traces, frames, n, len, h->r.slot_bytes(), SSPSD_MEM_HOST, loss, info);
}

}  // extern "C"
