    	this.myAmount = myAmount;
		myRandom = ThreadLocalRandom.current();
		this.multiplier = multiplier;
