// Device-resident storage behind flan::AudioBuffer / flan::PVBuffer in the B200 build.
//
// The reference's buffers are std::vector<Sample> / std::vector<MF> with reference-returning accessors
// (AudioBuffer.h:190,212-213; PVBuffer.h:250,272-273). Here every buffer is a host std::vector plus a device block
// with validity flags: conversions consume and produce the device copy; any host accessor lazily downloads it (or
// awaits a download that the producing call already started); any mutable host accessor invalidates the device copy.
// A chain such as
//     audio.convert_to_PV().convert_to_audio()
// therefore never moves the PV data across PCIe, and nothing on it calls cudaMalloc, cudaFree or a stream-wide
// synchronise in the steady state:
//   * device blocks come from the engine's block cache (flan_b200_malloc / _free);
//   * host vectors of buffers that die are recycled through a process-wide pool (same element count -> same vector, no
//     84 ms of page faults for a fresh 230 MB std::vector), and a vector that keeps coming back is page-locked once
//     (cudaHostRegister) so that later copies into and out of it are asynchronous DMA at PCIe speed;
//   * uploads and downloads run on the engine's copy streams, ordered against kernels per block, and a host accessor
//     waits for exactly its own buffer (flan_b200_wait).
#pragma once

#include <atomic>
#include <cstddef>
#include <cstdint>
#include <functional>
#include <memory>
#include <mutex>
#include <vector>

struct flan_b200_ctx;
struct flan_b200_multi;

namespace flan::b200 {

// Process-wide engine context (device from $FLAN_B200_DEVICE, default 0). Returns nullptr and prints the reason
// when no CUDA device / library is usable: there is no CPU fallback.
flan_b200_ctx * context();

// Every visible GPU behind one handle (include/flan_b200.h: flan_b200_multi_*), or nullptr when the process uses a
// single device: $FLAN_B200_DEVICE names one, or only one is visible. $FLAN_B200_DEVICES="0,1,..." picks a subset.
// When it exists, context() is its device 0. Long signals are then cut into frame-range shards, one per GPU, by
// Audio::convert_to_PV, PV::repitch / stretch / modify_time keep them sharded (a per-bin or descending time map
// gathers onto device 0), and PV::convert_to_audio resynthesises them with the phase-state and halo exchange between
// the devices; the result is the single-device result bit for bit.
flan_b200_multi * multi();

// A PV that lives as frame-range shards on several devices (defined in b200_storage.cpp; owns the device blocks).
struct ShardedStore;
std::shared_ptr<ShardedStore> new_sharded_store();
void * sharded_descriptor( ShardedStore & );      // flan_b200_sharded_pv * (include/flan_b200.h)
// The call that wrote the shards also left their phase summaries on every device (flan_b200_multi_stretch /
// _modify_time): a resynthesis of the shards as they are may say so (flan_b200_multi_promise_unchanged). A mutable host
// access drops the shards, so a store that still exists still holds the rows that call wrote.
void set_sharded_summaries( ShardedStore & );
bool sharded_summaries( const ShardedStore & );

// Recycled host vectors (see the header comment). `pinned` reports whether the vector's storage is page-locked.
template<typename T> std::vector<T> pool_take( size_t count, bool zeroed, bool * pinned, bool only_if_pooled = false );
template<typename T> void pool_give( std::vector<T> && v, bool pinned );

template<typename T>
class Mirror
	{
public:
	Mirror() = default;
	explicit Mirror( size_t count );                                     // zero-filled host copy (reference: zero-initialised vector)
	Mirror( std::vector<T> && v ) : host_( std::move( v ) ), count_( host_.size() ) {}
	Mirror( Mirror && o ) noexcept { take( o ); }
	Mirror & operator=( Mirror && o ) noexcept { if( this != &o ) { release(); take( o ); } return *this; }
	Mirror( const Mirror & ) = delete;
	Mirror & operator=( const Mirror & ) = delete;
	~Mirror() { release(); }

	size_t size() const { return count_; }
	bool empty() const { return count_ == 0; }

	// Host view. The const form downloads (or awaits the producer's download) if the device copy is newer; the mutable
	// form also drops the device copy. Concurrent const access from several threads is safe, as it is for the
	// reference's plain vectors.
	const std::vector<T> & host() const { if( !host_valid_.load( std::memory_order_acquire ) ) sync_to_host(); return host_; }
	std::vector<T> & host_mut();

	// Device view (uploads if the host copy is newer). nullptr on failure.
	const T * device() const { return device_with( nullptr ); }
	// The same, but when an upload is needed `uploader( h, d )` performs it (e.g. pipelined with the kernels that consume
	// the data) instead of a plain copy; *uploaded reports whether it ran. uploader returns a flan_b200 status code.
	const T * device_with( const std::function<int( const T * h, T * d )> * uploader, bool * uploaded = nullptr ) const;

	// Fresh device block of `count` elements whose contents the caller is about to produce on the GPU. When h_prefetch
	// is given and the pool holds a vector of that size, *h_prefetch is its storage: the caller's call also copies the
	// result there (asynchronously), and the host accessors only wait for that copy. nullptr otherwise.
	static Mirror device_result( size_t count, T ** d_out, T ** h_prefetch = nullptr );
	// Where the producing call reports the is_nan_or_inf() pre-scan (printed, like AudioPV.cpp:88-89, by the first host access)
	void set_nan_flag( const volatile int * flag ) { nan_flag_ = flag; }
	// A host vector that came from pool_take (its page-locked state travels with it).
	static Mirror adopt_host( std::vector<T> && v, bool pinned );
	// Storage sharded over several devices: host accessors gather it, device() gathers it onto device 0.
	static Mirror from_shards( size_t count, std::shared_ptr<ShardedStore> shards );
	const std::shared_ptr<ShardedStore> & shards() const { return shards_; }
	// The host vector holds the newest copy (a multi-device scatter reads it directly).
	bool host_is_current() const { return host_valid_.load( std::memory_order_acquire ); }
	const T * host_data_if_current() const { return host_is_current() ? host_.data() : nullptr; }

	// The device copy is still exactly what the call that produced it wrote (never re-uploaded from the host): phase
	// summaries that call left in the engine (flan_b200_modify_time) describe it (flan_b200_promise_unchanged).
	bool device_untouched() const { return produced_on_device_ && uploads_ == 0 && device_valid_.load( std::memory_order_acquire ); }

	Mirror deep_copy() const;

private:
	struct DeviceMem;
	void sync_to_host() const;
	void release();
	void maybe_pin_host() const;
	void take( Mirror & o );

	mutable std::vector<T> host_;
	size_t count_ = 0;
	mutable std::atomic<bool> host_valid_{ true };
	mutable std::atomic<bool> device_valid_{ false };
	mutable std::shared_ptr<DeviceMem> dev_;
	mutable std::shared_ptr<ShardedStore> shards_;
	mutable std::mutex lazy_;              // serialises the lazy upload / download
	mutable bool host_pinned_ = false;     // host_'s storage is page-locked (pooled vector or registered here)
	mutable const T * pinned_ptr_ = nullptr;   // the range that was registered (a user may have reallocated the vector since)
	mutable bool download_in_flight_ = false;  // the producer started an asynchronous copy into host_
	mutable bool upload_in_flight_ = false;    // an asynchronous copy out of (page-locked) host_ may still be running
	mutable int uploads_ = 0;
	bool produced_on_device_ = false;
	mutable const volatile int * nan_flag_ = nullptr;
	};

}
